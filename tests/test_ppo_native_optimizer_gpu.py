"""Each optimiser step of the native PPO update (taco_ppo_apply: gradient norm, clip, Adam, spectral projection, bf16 re-pack)
against float64 references: ``nn.utils.clip_grad_norm_`` and ``torch.optim.Adam(eps=1e-5)`` on float64 copies of the kernel's own
pre-step state and gradient (``make_optimizer`` and ``ppo_update`` of taco_b200.ppo), and ``torch.linalg.matrix_norm(ord=2)`` for
the projection.  GPU only.

The steps are driven one at a time through the C ABI (begin_update -> forward_loss -> decide -> backward -> apply).  Between
backward and apply a test may overwrite the gradient on the current stream, as the data-parallel path does with its all-reduce.

Bars (every test prints its measured maxima next to them):
  * Adam moments m, v: <= 1e-6 x max|ref| per tensor (one fp32 FMA chain);
  * the parameter step d = p_new - p_old, per element: |d - d_ref| <= 1e-4 |d_ref| + 1 ulp(p_old) + s(m).  The bias corrections
    come from powf(0.999f, t), and 0.999f is 1.3e-5 off 0.999 (6.5e-6 on the step at t = 1); the final subtraction rounds to
    fp32.  s(m) is the step error of rounding m's two terms to fp32, 2.5e-7 (0.9 |m_old| + 0.1 |g|) / (sqrt(v_hat) + eps) times
    the step size: where the two terms cancel, no fp32 Adam can do better;
  * gradient norm and clip coefficient (log columns 5 and 7): <= 1e-6 relative; the step counter exactly;
  * `world` identical ranks emulated in one process (loss sums and gradient multiplied by world): bitwise equal to world 1;
  * after a projection: ||W||_2 <= c (1 + 1e-3) and sigma_true (1 - 1e-3) <= sigmas() <= sigma_true (1 + 1e-5).  Power
    iteration only underestimates sigma; stopping on a change threshold eps leaves an error of about min(gap, eps / (2 gap)), at
    most sqrt(eps / 2) = 7e-4 for the kernel's eps = 1e-6.  A start vector with almost no weight on the top singular vector can
    still stop on sigma_2; with a top gap of 1e-3 that is within the bar by construction, which is why the gap is not smaller.
    When sigmas() > c, W == fp32(W fp32(c / sigma)) bitwise, otherwise
    W is bitwise unchanged, and every other parameter is bitwise unchanged either way;
  * the bf16 operand copies: the next forward is bitwise that of a fresh handle loaded with the same parameters, and a whole
    update is bitwise the same with a device synchronisation after every library call.
"""
import copy
import ctypes as C
import types

import numpy as np
import pytest
import torch

from test_ppo_native_gpu import _golden_cfg, _hyper
from test_ppo_native_stacked_gpu import _stacked_setup

pytestmark = pytest.mark.gpu

F32 = lambda x: float(np.float32(x))


def _flat(buf):
    f = lambda t: t.reshape(-1, *t.shape[2:]).contiguous()
    obs = f(buf.obs_buf)
    return {"obs": obs.reshape(obs.shape[0], -1), "states": f(buf.states_buf), "act": buf.act_buf.reshape(-1, buf.act_buf.size(-1)).contiguous(),
            "logp": buf.logp_buf.reshape(-1).contiguous(), "adv": buf.adv_buf.reshape(-1).contiguous(), "ret": buf.ret_buf.reshape(-1).contiguous()}


def _setup(actor_hidden, critic_hidden=(32,), layers=1, obs_dim=26, n_total=256, n_mb=2, seed=0):
    """An agent and a rollout whose old log-probabilities come from the agent itself; n_mb minibatches of n_total / n_mb samples."""
    from taco_b200.ppo import TorchActorCritic
    torch.manual_seed(seed)
    agent = TorchActorCritic(obs_dim, 4, list(actor_hidden), 26, 64, list(critic_hidden), lstm_layers=layers).cuda()
    gen = torch.Generator(device="cuda").manual_seed(seed)
    rnd = lambda *s: torch.randn(*s, device="cuda", generator=gen)
    buf = types.SimpleNamespace(obs_buf=rnd(1, n_total, 1, obs_dim) * 0.5, states_buf=rnd(1, n_total, 5, 26) * 0.5,
                                act_buf=rnd(1, n_total, 4).clamp(-1, 1), ret_buf=rnd(1, n_total, 1) * 0.3, adv_buf=rnd(1, n_total, 1))
    with torch.no_grad():
        logp = agent.evaluate(buf.obs_buf.view(-1, 1, obs_dim), buf.states_buf.view(-1, 5, 26), buf.act_buf.view(-1, 4))[0]
        buf.logp_buf = (logp + 0.05 * torch.randn(logp.shape, device="cuda", generator=gen)).view(1, n_total, 1)
        buf.value_buf = torch.zeros(1, n_total, 1, device="cuda")
    return agent, buf, list(torch.randperm(n_total, device="cuda", generator=gen).view(n_mb, -1))


class _Steps:
    """One NativePPO handle driven one optimiser step at a time through the C ABI."""

    def __init__(self, agent, buf, batch):
        from taco_b200.ppo_native import NativePPO
        self.d = _flat(buf)
        self.nat = NativePPO(agent, batch)
        self.nat._create(self.d["states"].shape[1])

    def begin(self):
        from taco_b200 import _capi
        _capi.check(self.nat._lib.taco_ppo_begin_update(self.nat._h, self.nat._stream()), "begin")

    def forward(self, hy, idx):
        from taco_b200 import _capi
        d, p = self.d, (lambda t: C.c_void_p(t.data_ptr()))
        _capi.check(self.nat._lib.taco_ppo_forward_loss(self.nat._h, C.byref(hy), p(d["obs"]), p(d["states"]), p(d["act"]), p(d["logp"]), p(d["adv"]),
                                                        p(d["ret"]), p(idx), self.nat._stream()), "forward_loss")

    def step(self, hy, idx, grad=None, world=1, after_forward=None):
        """One optimiser step; returns the state it started from (parameters, moments, step counter, the gradient apply reads)."""
        from taco_b200 import _capi
        nat, L, s = self.nat, self.nat._lib, self.nat._stream()
        self.forward(hy, idx)
        if after_forward is not None:
            after_forward()
        if world != 1:
            nat.loss_sums.mul_(world)
        _capi.check(L.taco_ppo_decide(nat._h, C.byref(hy), s), "decide")
        _capi.check(L.taco_ppo_backward(nat._h, s), "backward")
        if grad is not None:
            nat.grad.copy_(grad)
        if world != 1:
            nat.grad.mul_(world)
        pre = {"p": nat.params.clone(), "m": nat.adam_m.clone(), "v": nat.adam_v.clone(), "g": nat.grad.clone(), "step": int(nat.step.item())}
        _capi.check(L.taco_ppo_apply(nat._h, C.byref(hy), s), "apply")
        return pre

    def end(self, max_rows=64):
        from taco_b200 import _capi
        log = np.zeros((max_rows, 8), dtype=np.float32)
        n, steps, stop = C.c_int32(), C.c_int32(), C.c_int32()
        _capi.check(self.nat._lib.taco_ppo_end_update(self.nat._h, log.ctypes.data_as(C.c_void_p), max_rows, C.byref(n), C.byref(steps), C.byref(stop),
                                                      self.nat._stream()), "end_update")
        torch.cuda.synchronize()
        return log[:n.value], int(steps.value), bool(stop.value)

    def state(self):
        torch.cuda.synchronize()
        return {"p": self.nat.params.clone(), "m": self.nat.adam_m.clone(), "v": self.nat.adam_v.clone(), "step": int(self.nat.step.item())}


def _ref_step(nat, pre, hy):
    """clip_grad_norm_ + torch.optim.Adam(eps=1e-5) in float64 from the kernel's pre-step state: per tensor name p, m, v, and the
    total norm and clip coefficient."""
    v = lambda flat: {n: t.double().cpu() for n, t in nat._views(flat).items()}
    p0, m0, v0, g0 = v(pre["p"]), v(pre["m"]), v(pre["v"]), v(pre["g"])
    prm = {n: torch.nn.Parameter(p0[n].clone()) for n in p0}
    for n, t in prm.items():
        t.grad = g0[n].clone()
    max_grad = F32(hy.max_grad)
    norm = float(torch.nn.utils.clip_grad_norm_(list(prm.values()), max_grad))
    clipped = {n: t.grad.clone() for n, t in prm.items()}
    opt = torch.optim.Adam(list(prm.values()), lr=F32(hy.lr), eps=1e-5)
    for n, t in prm.items():
        opt.state[t] = {"step": torch.tensor(float(pre["step"])), "exp_avg": m0[n].clone(), "exp_avg_sq": v0[n].clone()}
    opt.step()
    out = {n: {"p": t.detach(), "m": opt.state[t]["exp_avg"], "v": opt.state[t]["exp_avg_sq"], "p0": p0[n], "m0": m0[n], "g": clipped[n]}
           for n, t in prm.items()}
    return out, norm, min(max_grad / (norm + 1e-6), 1.0), pre["step"] + 1


def _check_adam(nat, ref, t, lr, post, names, worst):
    """m, v, and the parameter step of the tensors `names` against the float64 step; accumulates the worst ratios error / bar."""
    p1, m1, v1 = ({n: x.double().cpu() for n, x in nat._views(post[k]).items()} for k in ("p", "m", "v"))
    bc1, bc2 = 1 - 0.9 ** t, 1 - 0.999 ** t
    for n in ref:
        r = ref[n]
        for key, got in (("m", m1[n]), ("v", v1[n])):
            scale = float(r[key].abs().max())
            err = float((got - r[key]).abs().max())
            worst[key] = max(worst[key], err / scale if scale > 0 else (0.0 if err == 0 else float("inf")))
        if n not in names:
            continue
        d, d_ref = p1[n] - r["p0"], r["p"] - r["p0"]
        ulp = torch.from_numpy(np.spacing(np.abs(r["p0"].numpy().astype(np.float32))).astype(np.float64))
        denom = (r["v"] / bc2).sqrt() + 1e-5
        s_m = (lr / bc1) * 2.5e-7 * (0.9 * r["m0"].abs() + 0.1 * r["g"].abs()) / denom
        bar = 1e-4 * d_ref.abs() + ulp + s_m
        ratio = float(((d - d_ref).abs() / bar).max())
        worst["step"] = max(worst["step"], ratio)
        worst["step_rel"] = max(worst["step_rel"], float(((d - d_ref).abs() - ulp - s_m).clamp(min=0).div(d_ref.abs().clamp(min=1e-30)).max()))


def _spread(n, gen, norm):
    """A gradient whose elements spread over 1e-9 .. 1e2 in magnitude (random signs) before it is scaled to the given norm."""
    mag = 10.0 ** (torch.rand(n, generator=gen, dtype=torch.float64) * 11.0 - 9.0)
    sign = torch.where(torch.rand(n, generator=gen) < 0.5, -1.0, 1.0).double()
    g = mag * sign
    return (g * (norm / float(g.norm()))).float().cuda()


def _report(name, worst, bars):
    for k, b in bars.items():
        print(f"{name}: {k} max {worst[k]:.3e} (bar {b})")


# ------------------------------------------------------------------------------------------------ 1. clipping and Adam
@pytest.mark.parametrize("resume", [False, True])
def test_clip_and_adam_against_float64(resume):
    """Injected gradients, projection off: clip inactive / active (100 x max_grad) / a zero gradient after non-zero steps, elements
    over 1e-9 .. 1e2 so that some sit where sqrt(v_hat) meets eps.  resume: from a torch Adam state at step 1000 (load_from)."""
    from taco_b200.ppo import make_optimizer
    agent, buf, idx = _setup([64, 48], n_total=512)
    cfg = _golden_cfg(False, target_kl=1e9)
    hy = _hyper(cfg, 1e-3, 4.0)
    st = _Steps(agent, buf, idx[0].numel())
    t0 = 0
    if resume:
        gen = torch.Generator().manual_seed(7)
        opt = make_optimizer(agent, cfg)
        for prm in agent.parameters():
            m = torch.randn(prm.shape, generator=gen) * 1e-3
            opt.state[prm] = {"step": torch.tensor(1000.0), "exp_avg": m.cuda(), "exp_avg_sq": (m * m * 2.0 + 1e-12).cuda()}
        st.nat.load_from(agent, opt)
        t0 = 1000
        assert int(st.nat.step.item()) == 1000
    n = st.nat.n_params
    gen = torch.Generator().manual_seed(11)
    mg = F32(hy.max_grad)
    plan = [("inactive", 0.5 * mg), ("active", 100 * mg), ("inactive", 0.25 * mg), ("zero", 0.0), ("active", 100 * mg)]
    worst = {"m": 0.0, "v": 0.0, "step": 0.0, "step_rel": 0.0, "norm": 0.0, "coef": 0.0}
    names = set(st.nat._names)
    for k, (kind, norm) in enumerate(plan):
        grad = torch.zeros(n, device="cuda") if kind == "zero" else _spread(n, gen, norm)
        st.begin()
        pre = st.step(hy, idx[k % len(idx)], grad=grad)
        log, steps, stop = st.end()
        assert not stop and len(log) == 1 and steps == t0 + k + 1
        ref, norm_ref, coef_ref, t = _ref_step(st.nat, pre, hy)
        assert (coef_ref < 1.0) == (kind == "active")
        _check_adam(st.nat, ref, t, F32(hy.lr), st.state(), names, worst)
        worst["norm"] = max(worst["norm"], abs(float(log[0, 5]) - norm_ref) / max(norm_ref, 1e-30) if norm_ref > 0 else float(log[0, 5]))
        worst["coef"] = max(worst["coef"], abs(float(log[0, 7]) - coef_ref) / coef_ref)
    _report(f"clip+adam resume={resume}", worst, {"m": 1e-6, "v": 1e-6, "step": "1 (error / bar)", "step_rel": 1e-4, "norm": 1e-6, "coef": 1e-6})
    assert worst["m"] <= 1e-6 and worst["v"] <= 1e-6 and worst["step"] <= 1.0
    assert worst["norm"] <= 1e-6 and worst["coef"] <= 1e-6
    st.nat.close()


# ------------------------------------------------------------------------------------------------ 2. data-parallel arithmetic
@pytest.mark.parametrize("lip", [False, True])
def test_world_ranks_in_one_process_are_bitwise_world_one(lip):
    """world identical ranks: the all-reduced loss sums and gradient are world x one rank's.  Every scaling is a power of two, so
    world 2 and 4 must reproduce world 1 bit for bit, early-stop decision included."""
    agent, buf, idx = _stacked_setup(layers=1)
    cfg = _golden_cfg(lip, target_kl=1e9)

    def run(world, target_kl, steps=8):
        hy = _hyper(cfg, 3e-3, 1.2)
        hy.target_kl, hy.world = target_kl, world
        st = _Steps(agent, buf, idx[0].numel())
        st.begin()
        for k in range(steps):
            st.step(hy, idx[k % len(idx)], world=world)
        log, n_steps, stop = st.end()
        s = st.state()
        out = (s["p"], s["m"], s["v"], s["step"], log, n_steps, stop, st.nat.sigmas() if lip else None)
        st.nat.close()
        return out

    base = run(1, 1e9)
    kl = base[4][:, 4]
    # a target whose 1.5 x lies between the KL of some minibatch r >= 1 and every KL before it: the stop fires at row r
    r = next((i for i in range(1, len(kl)) if kl[i] > kl[:i].max()), None)
    assert r is not None, kl
    target = float((kl[:r].max() + kl[r]) / 2 / 1.5)
    for target_kl in (1e9, target):
        ref = run(1, target_kl)
        if target_kl != 1e9:
            assert ref[6] and len(ref[4]) == r + 1 and ref[5] == r, (ref[4][:, 4], r)
        for world in (2, 4):
            got = run(world, target_kl)
            assert all(torch.equal(a, b) for a, b in zip(got[:3], ref[:3])), (world, target_kl)
            assert got[3] == ref[3] and got[5] == ref[5] and got[6] == ref[6] and np.array_equal(got[4], ref[4]), (world, target_kl)
            if lip:
                assert np.array_equal(got[7], ref[7])
    print(f"world 2 / 4 bitwise world 1 (projection {'on' if lip else 'off'}; early stop at row {r})")


# ------------------------------------------------------------------------------------------------ 3. spectral projection
def _svd_matrix(rows, cols, s, gen):
    U = torch.linalg.qr(torch.randn(rows, rows, generator=gen, dtype=torch.float64))[0]
    V = torch.linalg.qr(torch.randn(cols, cols, generator=gen, dtype=torch.float64))[0]
    k = min(rows, cols)
    return (U[:, :k] * torch.as_tensor(s[:k], dtype=torch.float64)) @ V[:, :k].T


def _spectrum(kind, rows, cols, init, gen):
    """An actor weight matrix of the given kind, scaled to sigma_1 = 1 (float64)."""
    k = min(rows, cols)
    if kind == "init":
        w = init.double()
    elif kind == "orth+noise":
        w = torch.nn.init.orthogonal_(torch.empty(rows, cols, dtype=torch.float64), gain=2 ** 0.5, generator=gen) \
            + 0.02 * torch.randn(rows, cols, generator=gen, dtype=torch.float64)
    elif kind == "gauss":
        w = torch.randn(rows, cols, generator=gen, dtype=torch.float64)
    else:
        gap = {"gap1e-1": 1e-1, "gap1e-2": 1e-2, "gap1e-3": 1e-3, "equal-top-two": 0.0}[kind]
        s = np.concatenate([[1.0, 1.0 - gap], np.linspace(0.8, 0.05, max(k - 2, 0))])
        w = _svd_matrix(rows, cols, s, gen)
    return w / torch.linalg.matrix_norm(w, ord=2)


def _actor_mats(nat):
    return [n for n in nat._names if n.startswith("actor_mlp") and n.endswith("weight")]


def _project_and_check(st, hy, idx, c, worst, label):
    """One optimiser step whose Adam part is a no-op (zero gradient, zero moments), then the projection bars on every actor matrix."""
    nat = st.nat
    torch.cuda.synchronize()
    nat.adam_m.zero_()
    nat.adam_v.zero_()
    before = nat.params.clone()
    mats = _actor_mats(nat)
    w0 = {n: t.clone() for n, t in nat._views(before).items()}
    st.begin()
    st.step(hy, idx, grad=torch.zeros_like(nat.grad))
    log, steps, stop = st.end()
    assert not stop
    after = nat.params.clone()
    sig = nat.sigmas()
    w1 = nat._views(after)
    for l, n in enumerate(mats):
        sv = torch.linalg.svdvals(w0[n].double())
        true = float(sv[0])
        s_rep = float(sig[l])
        assert s_rep <= true * (1 + 1e-5), (label, n, s_rep, true)
        worst["sigma_low"] = max(worst["sigma_low"], 1 - s_rep / true)
        if s_rep > c:
            sc = np.float32(c) / np.float32(s_rep)
            assert torch.equal(w1[n], w0[n] * torch.tensor(sc, device="cuda")), (label, n)
        else:
            assert torch.equal(w1[n], w0[n]), (label, n)
        norm = float(torch.linalg.matrix_norm(w1[n].double(), ord=2))
        worst["norm_over"] = max(worst["norm_over"], norm / c - 1)
        if 1 - s_rep / true > 1e-3 or norm > c * (1 + 1e-3):
            worst["fails"].append(f"{label} {n}: sigma {s_rep:.7f} true {true:.7f} (low by {1 - s_rep / true:.2e}), |W| / c - 1 = {norm / c - 1:.2e}")
    keep = torch.ones_like(before, dtype=torch.bool)
    for n, o in zip(nat._names, nat._offsets):
        if n in mats:
            keep[o:o + w0[n].numel()] = False
    assert torch.equal(after[keep], before[keep]), label


def _load_actor(agent, mats):
    with torch.no_grad():
        for lin, w in zip([m for m in agent.actor_mlp.layers if isinstance(m, torch.nn.Linear)], mats):
            lin.weight.copy_(w.float())


_SHAPES = {"golden": (26, [64, 48]), "bench": (26, [256, 256, 256]), "len_obs5": (130, [128, 128]), "wide_in": (256, [256, 16])}
_KINDS = ["init", "orth+noise", "gauss", "gap1e-1", "gap1e-2", "gap1e-3", "equal-top-two"]


@pytest.mark.parametrize("shape", list(_SHAPES))
def test_spectral_projection_cold_start(shape):
    """The handle's first projection, on matrices with sigma_1 = 1 and the spectra of _KINDS, for c below sigma_2 of every matrix,
    between sigma_2 and sigma_1, and above sigma_1."""
    obs_dim, hidden = _SHAPES[shape]
    worst = {"sigma_low": 0.0, "norm_over": -1.0, "fails": []}
    for ki, kind in enumerate(_KINDS):
        agent, buf, idx = _setup(hidden, obs_dim=obs_dim, n_total=256, seed=ki)
        lins = [m for m in agent.actor_mlp.layers if isinstance(m, torch.nn.Linear)]
        gen = torch.Generator().manual_seed(100 + ki)
        mats = [_spectrum(kind, m.out_features, m.in_features, m.weight.detach().cpu(), gen) for m in lins]
        s2 = [float(torch.linalg.svdvals(w)[1]) if min(w.shape) > 1 else 0.0 for w in mats]
        for c in (0.95 * min(s2), (1.0 + max(s2)) / 2, 1.05):
            _load_actor(agent, mats)
            st = _Steps(agent, buf, idx[0].numel())
            _project_and_check(st, _hyper(_golden_cfg(True, target_kl=1e9), 1e-3, c), idx[0], c, worst, f"{shape} {kind} c={c:.6f}")
            st.nat.close()
    print(f"{shape}: sigma below the SVD value by at most {worst['sigma_low']:.3e} (bar 1e-3); max |W|/c - 1 = {worst['norm_over']:.3e} (bar 1e-3)")
    assert not worst["fails"], worst["fails"]


def _orth_noise_actor(agent, seed):
    gen = torch.Generator().manual_seed(seed)
    lins = [m for m in agent.actor_mlp.layers if isinstance(m, torch.nn.Linear)]
    return [torch.nn.init.orthogonal_(torch.empty(m.out_features, m.in_features, dtype=torch.float64), gain=2 ** 0.5, generator=gen)
            + 0.02 * torch.randn(m.out_features, m.in_features, generator=gen, dtype=torch.float64) for m in lins]


@pytest.mark.parametrize("start", ["after_early_stop", "after_load_from"])
def test_spectral_projection_restarts(start):
    """after_early_stop: the first projection that runs follows an update whose first minibatch early-stopped (its projection
    launch returned at once).  after_load_from: a handle that has projected other weights is loaded with unrelated ones.  Either
    way the power iteration must start over as on a new handle; the benchmark's actor, orthogonal x sqrt(2) + 0.02 noise."""
    worst = {"sigma_low": 0.0, "norm_over": -1.0, "fails": []}
    c = 1.2
    for seed in range(3):
        agent, buf, idx = _setup([256, 256, 256], n_total=256, seed=seed)
        _load_actor(agent, _orth_noise_actor(agent, 10 + seed))
        st = _Steps(agent, buf, idx[0].numel())
        cfg = _golden_cfg(True, target_kl=1e9)
        if start == "after_early_stop":
            hy = _hyper(cfg, 1e-3, c)
            hy.target_kl = 1e-12
            st.begin()
            st.step(hy, idx[0], grad=torch.zeros_like(st.nat.grad))
            log, steps, stop = st.end()
            assert stop and steps == 0
        else:
            _project_and_check(st, _hyper(cfg, 1e-3, c), idx[0], c, worst, f"seed {seed} first weights")
            other = copy.deepcopy(agent)
            _load_actor(other, _orth_noise_actor(other, 50 + seed))
            st.nat.load_from(other)
        _project_and_check(st, _hyper(cfg, 1e-3, c), idx[1], c, worst, f"{start} seed {seed}")
        st.nat.close()
    print(f"{start}: sigma below the SVD value by at most {worst['sigma_low']:.3e} (bar 1e-3); max |W|/c - 1 = {worst['norm_over']:.3e} (bar 1e-3)")
    assert not worst["fails"], worst["fails"]


# ------------------------------------------------------------------------------------------------ 4. a real update, step by step
@pytest.mark.parametrize("layers", [1, 2])
def test_real_update_step_by_step(layers):
    """8 optimiser steps of 4096 samples, [256, 256, 256] MLPs, c = 1.2 (the projection scales every actor matrix at every step)."""
    agent, buf, idx = _setup([256, 256, 256], [256, 256, 256], layers=layers, n_total=16384, n_mb=4, seed=layers)
    c = 1.2
    hy = _hyper(_golden_cfg(True, target_kl=1e9), 1e-3, c)
    st = _Steps(agent, buf, idx[0].numel())
    mats = _actor_mats(st.nat)
    names = set(st.nat._names) - set(mats)
    worst = {"m": 0.0, "v": 0.0, "step": 0.0, "step_rel": 0.0, "norm": 0.0, "sigma_low": 0.0, "norm_over": -1.0}
    for k in range(8):
        st.begin()
        pre = st.step(hy, idx[k % len(idx)])
        log, steps, stop = st.end()
        assert not stop and steps == k + 1
        ref, norm_ref, coef_ref, t = _ref_step(st.nat, pre, hy)
        post = st.state()
        _check_adam(st.nat, ref, t, F32(hy.lr), post, names, worst)
        worst["norm"] = max(worst["norm"], abs(float(log[0, 5]) - norm_ref) / norm_ref)
        sig = st.nat.sigmas()
        w1 = st.nat._views(post["p"])
        for l, n in enumerate(mats):
            true = float(torch.linalg.matrix_norm(ref[n]["p"], ord=2))          # the float64 Adam result the projection acted on
            worst["sigma_low"] = max(worst["sigma_low"], 1 - float(sig[l]) / true)
            worst["norm_over"] = max(worst["norm_over"], float(torch.linalg.matrix_norm(w1[n].double(), ord=2)) / c - 1)
    _report(f"real update L={layers}", worst, {"m": 1e-6, "v": 1e-6, "step": "1 (error / bar)", "step_rel": 1e-4, "norm": 1e-6,
                                               "sigma_low": 1e-3, "norm_over": 1e-3})
    assert worst["m"] <= 1e-6 and worst["v"] <= 1e-6 and worst["step"] <= 1.0 and worst["norm"] <= 1e-6
    assert worst["sigma_low"] <= 1e-3 and worst["norm_over"] <= 1e-3
    st.nat.close()


# ------------------------------------------------------------------------------------------------ 5. re-pack and the asynchronous path
@pytest.mark.parametrize("layers", [1, 2])
@pytest.mark.parametrize("lip", [False, True])
def test_repacked_operands_equal_a_fresh_handle(layers, lip):
    """After each step the next forward (action mean, value) is bitwise that of a fresh handle loaded with a snapshot of the
    parameters: the bf16 copies apply rebuilds (the actor's on the side stream, the critic's and its LSTM layers' on the caller's)
    are the ones a fresh load builds."""
    from taco_b200 import _capi
    agent, buf, idx = _stacked_setup(layers=layers)
    hy = _hyper(_golden_cfg(lip, target_kl=1e9), 3e-3, 1.2)
    st = _Steps(agent, buf, idx[0].numel())
    fd = _Steps(agent, buf, idx[0].numel())
    fresh = fd.nat
    checked = []

    def compare(k):
        def hook():
            torch.cuda.synchronize()
            mean, value = (t.clone() for t in st.nat.debug_outputs())
            fresh.params.copy_(st.nat.params)
            _capi.check(fresh._lib.taco_ppo_params_changed(fresh._h, fresh._stream()), "params_changed")
            fd.begin()
            fd.forward(hy, idx[k % len(idx)])
            torch.cuda.synchronize()
            fm, fv = fresh.debug_outputs()
            assert torch.equal(mean, fm) and torch.equal(value, fv), (k, layers, lip)
            checked.append(k)
        return hook

    st.begin()
    for k in range(6):
        st.step(hy, idx[k % len(idx)], after_forward=compare(k) if k > 0 else None)
    st.end()
    assert checked == [1, 2, 3, 4, 5]
    print(f"L={layers} projection {'on' if lip else 'off'}: forward after each of 5 steps bitwise a fresh handle's")
    st.nat.close(); fresh.close()


class _SyncAfterEveryCall:
    """The library with a device synchronisation after every taco_* call."""

    def __init__(self, lib):
        self._lib = lib

    def __getattr__(self, name):
        fn = getattr(self._lib, name)
        if not name.startswith("taco_"):
            return fn

        def call(*args):
            rc = fn(*args)
            torch.cuda.synchronize()
            return rc
        return call


@pytest.mark.parametrize("layers", [1, 2])
def test_update_without_synchronisation_equals_synchronised(layers):
    """A whole nat.update (projection on: the actor's projection and re-pack run on the side stream) is bitwise the same update
    with torch.cuda.synchronize() after every library call."""
    from taco_b200.ppo_native import NativePPO
    agent, buf, idx = _stacked_setup(layers=layers)
    cfg = _golden_cfg(True, target_kl=1e9)
    res = []
    for sync in (False, True):
        nat = NativePPO(agent, idx[0].numel())
        if sync:
            nat._lib = _SyncAfterEveryCall(nat._lib)
        out = nat.update(buf, cfg, 10, batch_idx=idx)
        torch.cuda.synchronize()
        res.append((nat.params.clone(), nat.adam_m.clone(), nat.adam_v.clone(), int(nat.step.item()), out["log"].copy()))
        nat.close()
    (p0, m0, v0, s0, l0), (p1, m1, v1, s1, l1) = res
    assert s0 == s1 == cfg.train_iters * len(idx)
    assert torch.equal(p0, p1) and torch.equal(m0, m1) and torch.equal(v0, v1) and np.array_equal(l0, l1)
    print(f"L={layers}: asynchronous update bitwise the synchronised one ({s0} steps)")

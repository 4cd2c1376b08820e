"""The native PPO update with a stacked LSTM critic encoder (``nn.LSTM(state_dim, 64, L)``, L = 1..4; taco_ppo_create_layers).

Bars (the ones of tests/test_ppo_native_gpu.py, applied per layer):
  * the stacked bf16-operand emulation (tests/ppo_bf16_stacked.py, built on oracle/ppo_bf16.py) equals the one-layer emulation
    exactly for L = 1, and with its rounding switched off equals autograd to 5e-6 of every gradient's norm for L = 2 and 3 (CPU);
  * one layer through taco_ppo_create_layers is bit for bit taco_ppo_create: parameters, gradient, Adam moments and log rows of a
    whole update;
  * one minibatch, L = 2 and 3: action mean and value <= 2e-3 against the fp32 twin's ``evaluate``, loss sums at the existing
    relative tolerances, every gradient tensor (each ``*_lk`` included) within 1e-2 of its norm against the emulation at batch
    256, and within 2e-2 at batch 4096 with 256-wide MLPs.  At that shape the comparison sits at the emulation's own noise
    floor: perturbing the states by one part in 1e6 moves the emulation's critic gradients by 0.5-0.7 % of their norm, and
    the kernels' differences from it (fp32 accumulation order, the epilogue's exp-based gate functions) cross bf16 rounding
    and ReLU-mask boundaries in every layer.  Measured on a B200 with seeds 1 and 2: 0.4-0.7 % for one layer (the same as the
    perturbation), 1.0-1.5 % for two layers and 0.6-1.8 % for three; at batch 256 the two-layer critic is within 3e-4;
  * a whole update, L = 2, against the fp32 twin ``ppo_update`` on the same buffer and minibatches: the same optimiser-step
    count, logged losses / KL <= 2e-3 relative, update direction cosine >= 0.9 per group (actor, each LSTM layer, critic MLP)
    and >= 0.97 overall; the KL early stop leaves the parameters untouched;
  * round trip, L = 2: load_from / store_to return parameters and Adam state exactly, and after sync_rollout_nets_native the
    FP32 critic kernel reproduces the agent's critic to its usual 5e-6.
"""
import copy
import ctypes as C
import os
import types

import numpy as np
import pytest
import torch

import ppo_bf16_stacked as ps
from test_ppo_native_gpu import _golden, _golden_cfg, _hyper


def test_stacked_emulation_of_one_layer_is_the_one_layer_emulation():
    import oracle.ppo_bf16 as pb
    from taco_b200.ppo import TorchActorCritic
    torch.manual_seed(0)
    agent = TorchActorCritic(26, 4, [64, 48], 26, 64, [32])
    B = 256
    obs, states, act = torch.randn(B, 1, 26) * 0.7, torch.randn(B, 5, 26) * 0.7, torch.randn(B, 4).clamp(-1.5, 1.5)
    adv, ret, old = torch.randn(B), torch.randn(B) * 0.5, torch.randn(B)
    args = (obs, states, act, old, adv, ret, 0.2, 1.0, 0.5, 0.01)
    g1, s1 = pb.minibatch_grads(agent, *args)
    g2, s2 = ps.minibatch_grads(agent, *args)
    assert set(g1) == set(g2) and all(torch.equal(g1[n], g2[n]) for n in g1)
    assert torch.equal(s1["value"], s2["value"]) and torch.equal(s1["mean"], s2["mean"])


@pytest.mark.parametrize("layers", [2, 3])
def test_stacked_emulation_backprop_equals_autograd_without_rounding(layers):
    import oracle.ppo_bf16 as pb
    from taco_b200.ppo import TorchActorCritic
    torch.manual_seed(layers)
    agent = TorchActorCritic(26, 4, [64, 48], 26, 64, [32], lstm_layers=layers)
    with torch.no_grad():
        agent.log_std.fill_(-0.3)
    B = 256
    obs, states, act = torch.randn(B, 1, 26) * 0.7, torch.randn(B, 5, 26) * 0.7, torch.randn(B, 4).clamp(-1.5, 1.5)
    adv, ret = torch.randn(B), torch.randn(B) * 0.5
    with torch.no_grad():
        old = agent.evaluate(obs, states, act)[0] + 0.1 * torch.randn(B)
    logp, ent, value, mean, _ = agent.evaluate(obs, states, act)
    ratio = torch.exp(logp - old)
    loss = -torch.min(adv * ratio, adv * torch.clamp(ratio, 0.8, 1.2)).mean() + 0.5 * torch.nn.functional.mse_loss(ret.view(-1, 1), value) \
        + 0.01 * (-ent.mean())
    loss.backward()
    keep, pb.r = pb.r, (lambda x: x)
    try:
        g, _ = ps.minibatch_grads(agent, obs, states, act, old, adv, ret, 0.2, 1.0, 0.5, 0.01)
    finally:
        pb.r = keep
    names = [n for n, _ in agent.named_parameters()]
    assert sum(n.startswith("critic_encoder.") for n in names) == 4 * layers
    for n, prm in agent.named_parameters():
        assert float((g[n] - prm.grad).norm() / (prm.grad.norm() + 1e-12)) <= 5e-6, n


class _CreateOneLayer:
    """The library with taco_ppo_create_layers(..., 1, ...) answered by taco_ppo_create."""

    def __init__(self, lib):
        self._lib = lib

    def __getattr__(self, name):
        return getattr(self._lib, name)

    def taco_ppo_create_layers(self, device, cfg, layers, out):
        assert layers == 1
        return self._lib.taco_ppo_create(device, cfg, out)


@pytest.mark.gpu
def test_one_layer_through_create_layers_is_bitwise_create():
    from taco_b200.ppo import TorchActorCritic
    from taco_b200.ppo_native import NativePPO
    gg, init, final, buf, log = _golden("lip")
    idx = [row.tolist() for row in gg["idx"]]
    res = []
    for legacy in (False, True):
        agent = TorchActorCritic(26, 4, [64, 48], 26, 64, [32])
        agent.load_state_dict(init)
        agent.cuda()
        nat = NativePPO(agent, len(idx[0]))
        if legacy:
            nat._lib = _CreateOneLayer(nat._lib)
        out = nat.update(buf, _golden_cfg(True), int(gg["epoch"]), batch_idx=idx)
        torch.cuda.synchronize()
        res.append((nat.params.clone(), nat.grad.clone(), nat.adam_m.clone(), nat.adam_v.clone(), int(nat.step.item()), out["log"].copy()))
        nat.close()
    (p0, g0, m0, v0, s0, l0), (p1, g1, m1, v1, s1, l1) = res
    assert s0 == s1 == int(gg["optim_step"])
    assert torch.equal(p0, p1) and torch.equal(g0, g1) and torch.equal(m0, m1) and torch.equal(v0, v1)
    assert np.array_equal(l0, l1)


@pytest.mark.gpu
@pytest.mark.parametrize("layers", [2, 3])
@pytest.mark.parametrize("actor_hidden,critic_hidden,n_total,batch,seq", [
    ([64, 48], [32], 1024, 256, 5), ([256, 256, 256], [256, 256, 256], 8192, 4096, 5),
    ([64, 48], [32], 1024, 256, 1), ([64, 48], [32], 1024, 256, 8)])
def test_stacked_forward_losses_and_gradients_of_one_minibatch(layers, actor_hidden, critic_hidden, n_total, batch, seq):
    from taco_b200 import _capi
    from taco_b200.ppo import PPOConfig, TorchActorCritic
    from taco_b200.ppo_native import NativePPO
    torch.manual_seed(1)
    agent = TorchActorCritic(26, 4, actor_hidden, 26, 64, critic_hidden, lstm_layers=layers).cuda()
    with torch.no_grad():
        agent.log_std.fill_(-0.3)
    gen = torch.Generator(device="cuda").manual_seed(1)
    rnd = lambda *s: torch.randn(*s, device="cuda", generator=gen)
    obs, states, act = rnd(n_total, 1, 26) * 0.7, rnd(n_total, seq, 26) * 0.7, rnd(n_total, 4).clamp(-1.5, 1.5)
    adv, ret = rnd(n_total), rnd(n_total) * 0.5
    keep_tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False                     # the fp32 twin's LSTM in full fp32
    try:
        with torch.no_grad():
            old_logp = agent.evaluate(obs, states, act)[0] + 0.1 * rnd(n_total)
        idx = torch.randperm(n_total, device="cuda", generator=gen)[:batch]
        cfg = PPOConfig(target_kl=1e9, ent_coef=0.01)
        nat = NativePPO(agent, batch)
        nat._create(seq)
        hy = _hyper(cfg, 1e-3, 4.0)
        L, s, p = nat._lib, nat._stream(), (lambda t: C.c_void_p(t.data_ptr()))
        _capi.check(L.taco_ppo_begin_update(nat._h, s), "begin")
        _capi.check(L.taco_ppo_forward_loss(nat._h, C.byref(hy), p(obs.reshape(n_total, -1)), p(states), p(act), p(old_logp), p(adv), p(ret), p(idx), s), "fwd")
        torch.cuda.synchronize()
        sums = nat.loss_sums.clone()
        _capi.check(L.taco_ppo_decide(nat._h, C.byref(hy), s), "decide")
        _capi.check(L.taco_ppo_backward(nat._h, s), "bwd")
        torch.cuda.synchronize()
        mean_n, value_n = nat.debug_outputs()
        with torch.no_grad():
            logp, ent, value, mean, _ = agent.evaluate(obs[idx], states[idx], act[idx])
            ratio = torch.exp(logp - old_logp[idx])
            sur = -torch.min(adv[idx] * ratio, adv[idx] * torch.clamp(ratio, 1 - cfg.clip, 1 + cfg.clip)).mean()
            vl = torch.nn.functional.mse_loss(ret[idx].view(-1, 1), value)
            kl = ((ratio - 1) - (logp - old_logp[idx])).mean()
    finally:
        torch.backends.cudnn.allow_tf32 = keep_tf32
    assert float((mean_n - mean).abs().max()) <= 2e-3 and float((value_n - value.view(-1)).abs().max()) <= 2e-3
    assert float(sums[0] / batch) == pytest.approx(float(sur), rel=5e-3, abs=2e-5)
    assert float(sums[1] / batch) == pytest.approx(float(vl), rel=1e-3)
    assert float(sums[2] / batch) == pytest.approx(float(kl), rel=5e-3, abs=1e-6)
    g, st = ps.minibatch_grads(agent, obs[idx], states[idx], act[idx], old_logp[idx], adv[idx], ret[idx], cfg.clip, cfg.pi_coef, cfg.vf_coef, cfg.ent_coef)
    assert float((mean_n - st["mean"]).abs().max()) <= 2e-4 and float((value_n - st["value"]).abs().max()) <= 2e-4
    views = nat._views(nat.grad)
    assert set(views) == set(g) and all(f"critic_encoder.layers.weight_ih_l{k}" in g for k in range(layers))
    worst = {n: float((views[n] - g[n]).norm() / (g[n].norm() + 1e-12)) for n in g}
    assert max(worst.values()) <= (1e-2 if batch <= 256 else 2e-2), worst
    nat.close()


def _stacked_setup(layers=2, H=16, N=256, seed=3):
    """A TorchActorCritic with a stacked critic and a rollout buffer whose old log-probabilities come from the agent itself."""
    from taco_b200.ppo import TorchActorCritic
    torch.manual_seed(seed)
    agent = TorchActorCritic(26, 4, [64, 48], 26, 64, [32], lstm_layers=layers).cuda()
    gen = torch.Generator(device="cuda").manual_seed(seed)
    rnd = lambda *s: torch.randn(*s, device="cuda", generator=gen)
    buf = types.SimpleNamespace(obs_buf=rnd(H, N, 1, 26) * 0.5, states_buf=rnd(H, N, 5, 26) * 0.5, act_buf=rnd(H, N, 4).clamp(-1, 1),
                                ret_buf=rnd(H, N, 1) * 0.3, adv_buf=rnd(H, N, 1))
    with torch.no_grad():
        logp, _, value, _, _ = agent.evaluate(buf.obs_buf.view(-1, 1, 26), buf.states_buf.view(-1, 5, 26), buf.act_buf.view(-1, 4))
        buf.logp_buf = (logp + 0.05 * torch.randn(logp.shape, device="cuda", generator=gen)).view(H, N, 1)
        buf.value_buf = value.view(H, N, 1).clone()
    idx = list(torch.randperm(H * N, device="cuda", generator=gen).view(4, -1))
    return agent, buf, idx


@pytest.mark.gpu
def test_stacked_update_against_the_fp32_twin():
    from taco_b200.ppo import make_optimizer, ppo_update
    from taco_b200.ppo_native import NativePPO
    agent, buf, idx = _stacked_setup()
    init = {k: v.detach().cpu().clone() for k, v in agent.state_dict().items()}
    cfg, epoch = _golden_cfg(True), 10
    twin = copy.deepcopy(agent)
    keep_tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        ref = ppo_update(twin, make_optimizer(twin, cfg), buf, cfg, epoch, batch_idx=idx)
    finally:
        torch.backends.cudnn.allow_tf32 = keep_tf32
    nat = NativePPO(agent, idx[0].numel())
    out = nat.update(buf, cfg, epoch, batch_idx=idx)
    nat.store_to(agent)
    assert out["optim_steps"] == ref["optim_steps"] == cfg.train_iters * len(idx) and not out["early_stop"]
    for name in ("policy_gradient_loss", "value_loss", "entropy_loss", "sum_loss", "approx_kl"):
        assert out[name] == pytest.approx(ref[name], rel=2e-3, abs=2e-5), name
    sd = {k: v.detach().cpu() for k, v in agent.state_dict().items()}
    fin = {k: v.detach().cpu() for k, v in twin.state_dict().items()}
    cos = lambda keys: float(torch.nn.functional.cosine_similarity(torch.cat([(sd[k] - init[k]).flatten() for k in keys]),
                                                                   torch.cat([(fin[k] - init[k]).flatten() for k in keys]), dim=0))
    groups = {"actor": [k for k in sd if k.startswith("actor_mlp")], "critic": [k for k in sd if k.startswith("critic_mlp")], "all": list(sd)}
    for k in range(2):
        groups[f"lstm_l{k}"] = [n for n in sd if n.startswith("critic_encoder") and n.endswith(f"_l{k}")]
    cs = {g: cos(ks) for g, ks in groups.items()}
    assert min(v for g, v in cs.items() if g != "all") >= 0.9 and cs["all"] >= 0.97, cs
    # the KL early stop: the first minibatch's KL is above 1.5 * target, nothing moves
    agent2, buf2, idx2 = _stacked_setup()
    init2 = {k: v.detach().cpu().clone() for k, v in agent2.state_dict().items()}
    nat2 = NativePPO(agent2, idx2[0].numel())
    out2 = nat2.update(buf2, _golden_cfg(True, target_kl=1e-7), epoch, batch_idx=idx2)
    assert out2["early_stop"] and out2["optim_steps"] == 0 and len(out2["log"]) == 1 and out2["log"][0, 6] == 1.0
    nat2.store_to(agent2)
    for k, v in agent2.state_dict().items():
        assert torch.equal(v.cpu(), init2[k]), k
    nat.close(); nat2.close()


@pytest.mark.gpu
def test_stacked_round_trip_and_rollout_sync():
    import taco_b200
    from taco_b200.ppo import make_optimizer, sync_rollout_nets_native
    from taco_b200.ppo_native import NativePPO
    agent, buf, idx = _stacked_setup()
    cfg = _golden_cfg(False)
    nat = NativePPO(agent, idx[0].numel())
    out = nat.update(buf, cfg, 10, batch_idx=idx)
    assert out["optim_steps"] == cfg.train_iters * len(idx)
    opt = make_optimizer(agent, cfg)
    nat.store_to(agent, opt)
    sd = {k: v.detach().clone() for k, v in agent.state_dict().items()}
    nat2 = NativePPO(agent, idx[0].numel())
    nat2._create(5)
    nat2.load_from(agent, opt)
    assert torch.equal(nat2.params, nat.params) and torch.equal(nat2.adam_m, nat.adam_m) and torch.equal(nat2.adam_v, nat.adam_v)
    assert int(nat2.step.item()) == int(nat.step.item())
    opt2 = make_optimizer(agent, cfg)
    for p in agent.parameters():                                   # scribble over the module, then restore it from the native state
        p.data.add_(1.0)
    nat2.store_to(agent, opt2)
    for k, v in agent.state_dict().items():
        assert torch.equal(v, sd[k]), k
    for p in agent.parameters():
        st, st2 = opt.state[p], opt2.state[p]
        assert torch.equal(st["exp_avg"], st2["exp_avg"]) and torch.equal(st["exp_avg_sq"], st2["exp_avg_sq"]) and float(st["step"]) == float(st2["step"])
    # the FP32 rollout critic loads every layer straight from the flat parameter vector
    critic = taco_b200.CriticLSTM(26, 5, 64, [32], lstm_layers=2)
    sync_rollout_nets_native(nat2, critic=critic)
    states = buf.states_buf[0]
    v = critic.forward(states).cpu()
    cpu = copy.deepcopy(agent).cpu()
    with torch.no_grad():
        ref = cpu.critic_mlp(cpu.critic_encoder(states.cpu()))
    torch.testing.assert_close(v, ref, rtol=0, atol=5e-6)
    critic.close(); nat.close(); nat2.close()


def test_layer_count_outside_1_to_4_is_rejected_before_touching_the_device():
    from taco_b200 import _capi, build
    build.build()
    lib = _capi.lib()
    cfg = _capi.TacoPPOCfg(batch=256, obs_dim=26, act_dim=4, state_dim=26, seq_len=5, lstm_hidden=64, n_actor_hidden=1, n_critic_hidden=1)
    h = C.c_void_p()
    for layers in (0, 5, -1):
        assert lib.taco_ppo_create_layers(0, C.byref(cfg), layers, C.byref(h)) == -1
        assert b"lstm_layers" in lib.taco_last_error() and not h.value

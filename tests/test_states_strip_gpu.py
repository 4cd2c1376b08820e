"""The env-owned state history strip (taco_env_states_strip): each step writes only its newest frame, and the step that wraps the
window offset to 0 moves the kept frames to the start of the env's row.  GPU only.

The rollout ring (taco_env_attach_rollout) keeps the contiguous shift of the whole window, so an env stepping into a ring is the
contiguous reference: every window the strip shows must equal, bit for bit, the slot the ring path wrote for the same step --
across several rebases, with forced and natural resets next to them, for both launch shapes (at most one CTA per SM, and more)
and for env counts that are not a multiple of the CTA size."""
import ctypes as C

import pytest
import torch

pytestmark = pytest.mark.gpu

K = 16                      # the window period at len_states = 5


def _strip_period(env):
    base, frames, period = C.c_void_p(), C.c_int32(), C.c_int32()
    env._lib.taco_env_states_strip(env._h, C.byref(base), C.byref(frames), C.byref(period))
    return frames.value, period.value


def _force_resets(envs, step, n):
    if step in (K - 2, K - 1, K, 2 * K - 1, 2 * K + 1):      # next to each rebase, on both sides
        idx = torch.arange(step % 7, n, 97, device="cuda:0")
        for e in envs:
            e.reset_buf[idx] = 1


@pytest.mark.parametrize("task,n,dr", [("flip", 1000, False), ("flip", 24001, False), ("mix", 24001, True)])
def test_strip_matches_the_contiguous_ring_across_rebases(task, n, dr):
    from taco_b200 import FpvVecTask, RolloutBuffer, make_cfg
    steps = 2 * K + 3
    cfg = make_cfg(task, n, domain_randomization=dr, **{"env.maxEpisodeLength": 11})    # natural resets and time-outs in the window
    a = FpvVecTask(cfg, seed=9)
    b = FpvVecTask(cfg, seed=9)
    assert _strip_period(a) == (5 + K - 1, K)
    buf = RolloutBuffer(n, 26, 1, 26, 5, 4, steps, 1, 0.99, 0.95, "cuda:0")
    b.attach_rollout(buf)
    kept = None
    for t in range(steps):
        _force_resets((a, b), t, n)
        act = a.random_actions(t)
        o, r, x, e = a.step(act)
        b.step(act)
        st = o["states"]
        assert st.shape == (n, 5, 26) and st.stride() == ((5 + K - 1) * 26, 26, 1) and st.storage_offset() == ((t + 1) % K) * 26
        assert torch.equal(st, buf.states_ring[t + 1]), t
        assert torch.equal(o["obs"], buf.obs_ring[t + 1]) and torch.equal(r, buf.rew_buf[t, :, 0]), t
        if kept is not None:                                     # the previous step's window is left as it was
            assert torch.equal(kept[0], kept[1]), t
        kept = (st, st.clone())
    assert float(buf.done_buf.sum()) > 0
    b.detach_rollout()                                           # the ring's newest slot goes back into b's strip
    for t in range(steps, steps + K):
        act = a.random_actions(t)
        a.step(act); b.step(act)
        assert torch.equal(a.states_buf, b.states_buf), t
    a.close(); b.close()


def _critic(gen, hid=32, mlp=(64, 64)):
    from taco_b200 import CriticLSTM
    lstm = [(torch.randn(4 * hid, 26, generator=gen) * 0.3, torch.randn(4 * hid, hid, generator=gen) * 0.2,
             torch.randn(4 * hid, generator=gen) * 0.1, torch.randn(4 * hid, generator=gen) * 0.1)]
    cs = [hid] + list(mlp) + [1]
    cw = [torch.randn(cs[i + 1], cs[i], generator=gen) / cs[i] ** 0.5 for i in range(len(cs) - 1)]
    cb = [torch.randn(cs[i + 1], generator=gen) * 0.1 for i in range(len(cs) - 1)]
    c = CriticLSTM(26, 5, hid, list(mlp))
    c.load(lstm, cw, cb)
    return c, (lstm, cw, cb)


@pytest.mark.parametrize("tensor_cores", [False, True])
def test_critic_on_the_strip_window_matches_contiguous(tensor_cores):
    from taco_b200 import FpvVecTask, make_cfg
    n = 24001
    env = FpvVecTask(make_cfg("flip", n), seed=3)
    critic, _ = _critic(torch.Generator().manual_seed(4))
    for t in range(K + 2):                                       # odd and even window offsets, a rebase in between
        env.step(env.random_actions(t))
        view = env.states_buf
        assert not view.is_contiguous()
        got = critic.forward(view, tensor_cores=tensor_cores)
        assert torch.equal(got, critic.forward(view.contiguous(), tensor_cores=tensor_cores)), t
    env.close(); critic.close()


def test_graph_captured_steps_follow_the_device_offset():
    """Steps captured in a CUDA graph with no ring attached: the window offset comes from the device step counter, so replays of a
    3-step graph (not a divisor of the period) keep writing where eager steps would."""
    from taco_b200 import FpvVecTask, make_cfg
    n, H, reps = 5000, 3, 7
    cfg = make_cfg("rotate", n, **{"env.maxEpisodeLength": 13})
    a, b = FpvVecTask(cfg, seed=2), FpvVecTask(cfg, seed=2)
    acts = [a.random_actions(t) for t in range(H)]
    a.step(acts[0]); b.step(acts[0])
    torch.cuda.synchronize()
    b.graph_begin()
    base = b.step_count
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for s in range(H):
            b.step_raw(acts[s])
        b.graph_advance(H)
    b.step_count = base
    for r in range(reps):
        g.replay()
        b.step_count += H
        for s in range(H):
            a.step(acts[s])
        torch.cuda.synchronize()
        assert torch.equal(a.states_buf, b.states_buf), r
        assert torch.equal(a.obs_buf, b.obs_buf) and torch.equal(a.rew_buf, b.rew_buf), r
    b.graph_end()
    assert b.step_count == a.step_count == 1 + H * reps
    a.step(acts[1]); b.step(acts[1])
    assert torch.equal(a.states_buf, b.states_buf)
    a.close(); b.close()


def test_graphed_rollout_then_detach_continues_the_strip():
    """A GraphedRollout of horizon 5 (not a multiple of the period), replayed several times, equals the eager collect_rollout; after
    detaching, both envs continue in their strips from the same window."""
    from taco_b200 import ActorMLP, FpvVecTask, GraphedRollout, RolloutBuffer, collect_rollout, make_cfg
    n, H = 3000, 5
    gen = torch.Generator().manual_seed(6)
    sizes = [26, 64, 64, 4]
    aw = [torch.randn(sizes[i + 1], sizes[i], generator=gen) * 0.25 for i in range(3)]
    ab = [torch.zeros(sizes[i + 1]) for i in range(3)]
    critic, prm = _critic(gen, mlp=(64,))
    snaps = {}
    for mode in ("eager", "graph"):
        env = FpvVecTask(make_cfg("flip", n, **{"env.maxEpisodeLength": 9}), seed=8)
        actor = ActorMLP(26, [64, 64], 4)
        actor.load(aw, ab, log_std=torch.full((4,), -0.4))
        for t in range(3):
            env.step(env.random_actions(t))
        buf = RolloutBuffer(n, 26, 1, 26, 5, 4, H, 1, 0.99, 0.95, "cuda:0")
        out = []
        if mode == "eager":
            for _ in range(4):
                collect_rollout(env, actor, buf, critic, seed=1, tensor_cores=True)
                out.append((buf.states_ring.clone(), buf.value_buf.clone()))
        else:
            gr = GraphedRollout(env, actor, buf, critic, seed=1, tensor_cores=True)
            out.append((buf.states_ring.clone(), buf.value_buf.clone()))
            for _ in range(3):
                gr.run()
                torch.cuda.synchronize()
                out.append((buf.states_ring.clone(), buf.value_buf.clone()))
            gr.close()
        env.detach_rollout()
        assert env.step_count == 3 + 4 * H
        for t in range(K):
            o, _, _, _ = env.step(env.random_actions(100 + t))
            out.append((o["states"].clone(), critic.forward(env.states_buf, tensor_cores=True)))
        snaps[mode] = out
        env.close(); actor.close()
    for k, (x, y) in enumerate(zip(snaps["eager"], snaps["graph"])):
        assert torch.equal(x[0], y[0]) and torch.equal(x[1], y[1]), k
    critic.close()


@pytest.mark.parametrize("mode", ["mapped", "copy", "compact"])
def test_host_buffer_step_writes_the_strip(mode, monkeypatch):
    """The C ABI host-buffer steps (mapped: the kernel's host-buffer variant; copy: chunked launches over CTA ranges) keep the same
    strip as the device step, across a rebase."""
    from taco_b200 import FpvVecTask, make_cfg
    n = 70001                                                    # 547 CTAs: more than one chunk of the copy pipeline
    monkeypatch.setenv("TACO_HOST_MODE", "copy" if mode == "copy" else "mapped")
    cfg = make_cfg("flip", n, **{"env.maxEpisodeLength": 10})
    a, b = FpvVecTask(cfg, seed=4), FpvVecTask(cfg, seed=4)
    rew = torch.empty(n, dtype=torch.float32).pin_memory()
    reset = torch.empty(n, dtype=torch.int64).pin_memory()
    tout = torch.empty(n, dtype=torch.uint8).pin_memory()
    flags = torch.empty(n, dtype=torch.uint8).pin_memory()
    for t in range(K + 3):
        act = a.random_actions(t)
        _, r, x, _ = a.step(act)
        h_act = act.cpu().pin_memory()
        if mode == "compact":
            b.step_host_compact(h_act, rew, flags)
        else:
            b.step_host(h_act, rew, reset, tout)
        torch.cuda.synchronize()
        assert torch.equal(a.states_buf, b.states_buf), t
        assert torch.equal(r.cpu(), rew), t
    a.close(); b.close()

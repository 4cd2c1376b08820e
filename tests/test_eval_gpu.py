"""The evaluation path on the device (taco_b200.evaluate, taco_env_attach_episode_log, taco_env_record_state): the episode log
against a float32 host replay of the same definitions -- on the oracle's per-step states and on the env's own exported states --,
its consistency with taco_env_stats, the episode-start rule, the capacity, graph replay against the eager loop, the trajectory
recorder and the exclusion of rollout rings.  GPU only."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

RUN_TOL = 5e-4          # the drift bar of tests/test_glue_golden_gpu.py (kernel vs the oracle over a run)
f32 = np.float32


def _nrm(x, y, z):
    return np.sqrt((x * x + y * y) + z * z).astype(f32)          # float32, op by op, like the kernel


def _frame_from_export(env, st):
    return dict(pos=st[:, 0:3], quat=st[:, 3:7], linvel=st[:, 7:10], angvel=st[:, 10:13], tpos=st[:, 13:16], roll=st[:, 21],
                progress=st[:, 34].astype(np.int64), reset=st[:, 38].astype(np.int64), rew=env.rew_buf.cpu().numpy(),
                tout=env.timeout_buf.cpu().numpy())


def _frame_from_oracle(ref):
    import parity_util as pu
    s = pu.oracle_state(ref)
    return dict(pos=s["pos"], quat=s["quat"], linvel=s["linvel"], angvel=s["angvel"], tpos=s["tpos"], roll=s["roll_cont"][:, 0],
                progress=s["progress"][:, 0].astype(np.int64), reset=s["reset"][:, 0].astype(np.int64), rew=ref.rew_buf.numpy(),
                tout=ref.timeout_buf.numpy())


class LogReplay:
    """The episode log's definitions (include/taco_b200.h TacoEpisode) replayed on the host in float32."""

    def __init__(self, gids, task, live):
        from taco_b200.evaluate import EPISODE_DTYPE
        self.dtype = EPISODE_DTYPE
        self.gids, self.task = np.asarray(gids, np.int64), np.asarray(task)
        n = len(self.gids)
        self.live = np.asarray(live, bool).copy()
        self.acc = {k: np.zeros(n, f32) for k in ("ret", "pe", "sp", "tilt", "av", "roll0")}
        self.records = []
        self.done_ret = []              # per step: (done mask, ret at the end) -- what taco_env_stats adds

    def step(self, t, f):
        a = self.acc
        d = (f["pos"] - f["tpos"]).astype(f32)
        pe = _nrm(d[:, 0], d[:, 1], d[:, 2])
        sp = _nrm(*(f["linvel"][:, j] for j in range(3)))
        av = _nrm(*(f["angvel"][:, j] for j in range(3)))
        qx, qy = f["quat"][:, 0], f["quat"][:, 1]
        cz = (f32(1) - f32(2) * (qx * qx + qy * qy)).astype(f32)
        tilt = np.arccos(np.clip(cz, f32(-1), f32(1))).astype(f32)
        a["ret"] = (a["ret"] + f["rew"].astype(f32)).astype(f32)
        a["pe"] = (a["pe"] + pe).astype(f32)
        a["sp"] = (a["sp"] + sp).astype(f32)
        a["tilt"] = np.maximum(a["tilt"], tilt)
        a["av"] = np.maximum(a["av"], av)
        flip = self.task == 2
        roll = np.where(flip, f["roll"], f32(0)).astype(f32)
        a["roll0"] = np.where(flip & (f["progress"] == 1), roll, a["roll0"]).astype(f32)
        done = f["reset"] != 0
        self.done_ret.append((done.copy(), a["ret"].copy()))
        for e in np.flatnonzero(done & self.live):
            ln = f32(f["progress"][e])
            r = np.zeros((), self.dtype)
            r["env_id"], r["end_step"], r["length"] = self.gids[e], t, f["progress"][e]
            r["task"], r["timed_out"] = self.task[e], int(f["tout"][e])
            r["ret"], r["pos_err_mean"], r["pos_err_final"] = a["ret"][e], a["pe"][e] / ln, pe[e]
            r["tilt_max"], r["speed_mean"], r["angvel_max"] = a["tilt"][e], a["sp"][e] / ln, a["av"][e]
            r["roll_travel"] = roll[e] - a["roll0"][e] if flip[e] else f32(0)
            self.records.append(r)
        for v in a.values():
            v[done] = 0
        self.live |= done

    def result(self):
        return np.array(self.records, dtype=self.dtype) if self.records else np.zeros(0, self.dtype)


def _sorted(recs):
    return recs[np.lexsort((recs["env_id"], recs["end_step"]))]


def _tasks(env):
    from taco_b200 import _capi
    gid = env.env_offset + np.arange(env.num_envs)
    mode = env.task_mode or env.cfg["task_mode"]
    if mode != "mix":
        return np.full(env.num_envs, _capi.TASK[mode])
    n1, n2 = int(env.num_envs_global / 3 * 1), int(env.num_envs_global / 3 * 2)
    return np.where(gid < n1, 0, np.where(gid < n2, 1, 2))


FLOATS = ("ret", "pos_err_mean", "pos_err_final", "tilt_max", "speed_mean", "angvel_max", "roll_travel")
INTS = ("env_id", "end_step", "length", "task", "timed_out")


def _assert_same_keys(got, want, where):
    assert len(got) == len(want), f"{where}: {len(got)} records, expected {len(want)}"
    for k in INTS:
        assert np.array_equal(got[k], want[k]), f"{where}: field {k} differs"


def _rel(a, b, floor):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float((np.abs(a - b) / np.maximum(np.abs(b), floor)).max()) if len(a) else 0.0


def _warp_sums(v):
    """The step kernel's warp butterfly of a float32 per-env vector (lane 0's value) per warp of 32 envs."""
    n = len(v)
    w = np.zeros(((n + 31) // 32) * 32, f32)
    w[:n] = v
    w = w.reshape(-1, 32)
    for o in (16, 8, 4, 2, 1):
        w = (w + w[:, np.arange(32) ^ o]).astype(f32)
    return w[:, 0]


@pytest.mark.parametrize("task", ["pos", "flip", "mix"])
def test_episode_log_against_oracle_env_states_and_stats(task):
    import parity_util as pu
    import taco_b200
    n, T = 512, 72
    cfg = taco_b200.make_cfg(task, n, domain_randomization=True)
    cfg["env"]["maxEpisodeLength"] = 25
    gpu, ref = pu.make_pair(cfg, debug_delay=False)
    gpu.reset()
    gpu.stats()                                                  # nothing stepped yet: clears nothing, starts the window
    log = taco_b200.EpisodeLog(gpu, 100000)
    gids, tasks = gpu.env_offset + np.arange(n), _tasks(gpu)
    from_oracle = LogReplay(gids, tasks, np.ones(n, bool))
    from_env = LogReplay(gids, tasks, np.ones(n, bool))
    finite = np.ones(n, bool)
    for t in range(T):
        a = pu.oracle_actions(ref, t)
        gpu.step(gpu.random_actions(t))
        ref.step(a)
        fo = _frame_from_oracle(ref)
        finite &= np.isfinite(fo["pos"]).all(1) & np.isfinite(fo["angvel"]).all(1) & ~ref.overflow.numpy()
        from_oracle.step(t, fo)
        from_env.step(t, _frame_from_export(gpu, gpu.export_state()))
    got = _sorted(log.read())
    assert log.dropped == 0 and len(got) > n                     # many time-outs and terminations inside the run
    assert got["timed_out"].any() and not got["timed_out"].all()
    # 1. the oracle's states: integers exact, floats within the drift bar (envs that stayed finite)
    want = _sorted(from_oracle.result())
    _assert_same_keys(got, want, f"{task} vs oracle")
    m = finite[got["env_id"] - gpu.env_offset]
    assert m.mean() > 0.95
    for k in FLOATS:
        floor = 1e-2 if k == "ret" else 1.0
        assert _rel(got[k][m], want[k][m], floor) <= RUN_TOL, f"{task} vs oracle: {k}"
    # 2. the env's own exported states: ret bit-identical, the rest within 1e-6 relative
    want = _sorted(from_env.result())
    _assert_same_keys(got, want, f"{task} vs export_state")
    assert np.array_equal(got["ret"].view(np.uint32), want["ret"].view(np.uint32))
    for k in FLOATS[1:]:
        assert _rel(got[k], want[k], 1e-3) <= 1e-6, f"{task} vs export_state: {k}"
    # 3. consistency with taco_env_stats over the same steps
    s = gpu.stats().cpu().numpy()
    assert len(got) == s[1] and int((got["timed_out"] != 0).sum()) == s[2]
    assert int(got["length"].astype(np.int64).sum()) == s[4]
    stats_ret = sum(float(_warp_sums(np.where(d, r, f32(0))).astype(np.float64).sum()) for d, r in from_env.done_ret)
    assert abs(s[3] - stats_ret) <= 1e-12 * abs(stats_ret)
    assert abs(got["ret"].astype(np.float64).sum() - s[3]) <= 1e-5 * abs(s[3])   # the float32 warp sums of the stats round
    log.close()
    gpu.close()


def _run_with_log(env, steps, capacity=100000):
    import taco_b200
    log = taco_b200.EpisodeLog(env, capacity)
    for _ in range(steps):
        env.step_raw(env.random_actions(env.step_count))
    return log


def test_episode_start_rule_attach_mid_run_and_reset_all():
    import taco_b200
    n, attach, reset = 1024, 13, 50
    cfg = taco_b200.make_cfg("flip", n, domain_randomization=True)
    cfg["env"]["maxEpisodeLength"] = 25
    env = taco_b200.FpvVecTask(cfg, "cuda:0", "cuda:0", -1, True, seed=11)
    for _ in range(attach):                                      # most envs are mid-episode when the log is attached
        env.step_raw(env.random_actions(env.step_count))
    log = taco_b200.EpisodeLog(env, 100000)
    replay = LogReplay(np.arange(n), _tasks(env), env.export_state()[:, 38] != 0)
    parts = []
    for k in range(attach, 80):
        if k == reset:                                           # every env mid-episode again: reset_all discards them
            parts.append((log.read(), replay.result(), attach))
            log.clear()
            env.reset_all()
            replay = LogReplay(np.arange(n), _tasks(env), np.ones(n, bool))
        t = env.step_count
        env.step_raw(env.random_actions(t))
        replay.step(t, _frame_from_export(env, env.export_state()))
    parts.append((log.read(), replay.result(), 0))
    for got, want, start in parts:
        got, want = _sorted(got), _sorted(want)
        assert len(got) > n // 2
        _assert_same_keys(got, want, f"window from step {start}")
        assert np.array_equal(got["ret"].view(np.uint32), want["ret"].view(np.uint32))   # no partial sum leaked into a record
        for k in FLOATS[1:]:
            assert _rel(got[k], want[k], 1e-3) <= 1e-6, k
        # every record is an episode that started inside the log's window (episodes already running are never recorded)
        assert np.all(got["length"] <= got["end_step"].astype(np.int64) - start + 1)
        # ... and every env that was mid-episode at the start of the window does get recorded after its first end
        assert len(np.unique(got["env_id"])) == n
    log.close()
    env.close()


def test_capacity_keeps_the_first_records_and_counts_the_dropped():
    import taco_b200
    n, steps, cap = 1024, 40, 300
    runs = []
    for capacity in (100000, cap):
        cfg = taco_b200.make_cfg("pos", n, domain_randomization=True)
        cfg["env"]["maxEpisodeLength"] = 25
        env = taco_b200.FpvVecTask(cfg, "cuda:0", "cuda:0", -1, True, seed=5)
        log = _run_with_log(env, steps, capacity=capacity)
        runs.append((log.read(), log.count, log.dropped))
        log.close()
        env.close()
    (full, n_full, d_full), (part, n_part, d_part) = runs
    assert d_full == 0 and n_full == len(full) > cap
    assert n_part == n_full and d_part == n_full - cap and len(part) == cap
    # records are appended in step order (within a step in an unspecified order): the kept ones are the first `cap`
    last = part["end_step"].max()
    full_keys = {(int(r["env_id"]), int(r["end_step"])) for r in full}
    assert all((int(r["env_id"]), int(r["end_step"])) in full_keys for r in part)
    assert np.array_equal(np.sort(part["end_step"]), np.sort(full["end_step"])[:cap])
    assert (full["end_step"] < last).sum() <= cap
    fk = {(int(r["env_id"]), int(r["end_step"])): r.tobytes() for r in full}
    assert all(fk[(int(r["env_id"]), int(r["end_step"]))] == r.tobytes() for r in part)


def _actor(seed=3):
    import taco_b200
    gen = torch.Generator().manual_seed(seed)
    sizes = [26, 128, 128, 4]
    actor = taco_b200.ActorMLP(26, sizes[1:-1], 4)
    actor.load([torch.randn(sizes[i + 1], sizes[i], generator=gen) / sizes[i] ** 0.5 for i in range(3)],
               [torch.randn(sizes[i + 1], generator=gen) * 0.1 for i in range(3)])
    return actor


@pytest.mark.parametrize("tc", [False, True])
def test_graph_replay_matches_eager_loop_and_actions_are_the_actor_mean(tc):
    import taco_b200
    n = 1024
    cfg = taco_b200.make_cfg("mix", n, domain_randomization=True)
    cfg["env"]["maxEpisodeLength"] = 30
    env = taco_b200.FpvVecTask(cfg, "cuda:0", "cuda:0", -1, True, seed=21)
    actor = _actor()
    if tc and not actor.tensor_cores_available:
        pytest.skip("tcgen05 actor kernel unavailable")
    ids = [0, 5, 400, n - 1]
    kw = dict(tensor_cores=tc, record_env_ids=ids, steps_per_replay=8)
    rec_e, traj_e, sum_e = taco_b200.evaluate_policy(env, actor, 10**9, 48, graph=False, **kw)
    rec_g, traj_g, sum_g = taco_b200.evaluate_policy(env, actor, 10**9, 48, graph=True, **kw)
    assert len(rec_e) > n // 2
    assert _sorted(rec_e).tobytes() == _sorted(rec_g).tobytes()
    assert traj_e["data"].shape == (48, len(ids), 68) and np.array_equal(traj_e["step"], np.arange(48))
    assert traj_e["data"].tobytes() == traj_g["data"].tobytes()
    assert set(sum_e) == set(sum_g) == {"pos", "rotate", "flip"}            # summed in record order, which is unspecified
    for name in sum_e:
        assert sum_e[name] == pytest.approx(sum_g[name], rel=1e-9, nan_ok=True), name
    # the applied actions are ActorMLP.forward of the observation at each step
    env.reset_all()
    for t in range(48):
        mean = actor.forward(env.obs_buf, tensor_cores=tc)
        assert np.array_equal(traj_g["data"][t, :, 64:], mean[ids].cpu().numpy()), f"step {t}"
        env.step_raw(mean)
        assert np.array_equal(traj_g["data"][t, :, :64], env.export_state()[ids]), f"step {t}"
    with pytest.raises(ValueError, match="even"):
        taco_b200.evaluate_policy(env, actor, 10, 16, steps_per_replay=7)
    actor.close()
    env.close()


def test_recorder_rows_equal_export_state_on_a_shard():
    import taco_b200
    n, off, glob = 300, 1200, 2000                               # global ids 1200..1499 straddle the rotate / flip boundary 1333
    cfg = taco_b200.make_cfg("mix", n, domain_randomization=True)
    cfg["env"]["maxEpisodeLength"] = 20
    env = taco_b200.FpvVecTask(cfg, "cuda:0", "cuda:0", -1, True, env_offset=off, num_envs_global=glob, seed=8)
    ids = torch.tensor([0, 7, 132, 133, n - 1], dtype=torch.int32, device="cuda:0")
    log = taco_b200.EpisodeLog(env, 10000)
    out = torch.empty(len(ids), 64, device="cuda:0")
    for t in range(30):
        env.step_raw(env.random_actions(t))
        env.record_state(ids, out=out)
        assert out.cpu().numpy().tobytes() == env.export_state()[ids.cpu().numpy()].tobytes(), f"step {t}"
    bad = env.record_state(torch.tensor([-1, n], dtype=torch.int32, device="cuda:0"))
    assert torch.isnan(bad).all()
    recs = log.read()
    assert len(recs) > 0
    assert np.array_equal(recs["task"], np.where(recs["env_id"] < int(glob / 3 * 2), 1, 2))
    assert (recs["task"] == 1).any() and (recs["task"] == 2).any()
    assert recs["env_id"].min() >= off and recs["env_id"].max() < off + n
    log.close()
    env.close()


def test_log_and_rollout_ring_exclude_each_other():
    import taco_b200
    n = 256
    env = taco_b200.FpvVecTask(taco_b200.make_cfg("pos", n), "cuda:0", "cuda:0", -1, True)
    buf = taco_b200.RolloutBuffer(n, 26, env.len_obs, 26, env.len_states, 4, 4, 1, 0.99, 0.95, "cuda:0")
    log = taco_b200.EpisodeLog(env, 100)
    with pytest.raises(RuntimeError, match="episode log"):
        env.attach_rollout(buf)
    log.close()
    env.attach_rollout(buf)
    with pytest.raises(RuntimeError, match="rollout ring"):
        taco_b200.EpisodeLog(env, 100)
    with pytest.raises(ValueError, match="rollout ring"):
        taco_b200.evaluate_policy(env, _actor(), 10, 16)
    env.detach_rollout()
    log = taco_b200.EpisodeLog(env, 100)
    log.clear()
    assert log.count == 0
    log.close()
    env.close()

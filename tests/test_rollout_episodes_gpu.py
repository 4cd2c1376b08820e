"""Training-time episode records and per-task summaries from the rollout ring (taco_b200.RolloutEpisodes,
taco_env_scan_rollout_episodes): the records against the episode log of a ring-free twin env, the summaries against
taco_env_stats and a float64 sum of the records, graph replays against the eager loop, the episode-start rule, the capacity, the
invalid calls and sharding.  GPU only."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

f32 = np.float32


def _rec_dtype():
    from taco_b200 import _capi
    return _capi.ROLLOUT_EPISODE_DTYPE


def _sorted(recs):
    return recs[np.lexsort((recs["env_id"], recs["end_step"]))]


def _first_six(log_records):
    """The first six fields of TacoEpisode records as TacoRolloutEpisode records."""
    dt = _rec_dtype()
    out = np.zeros(len(log_records), dt)
    for k in dt.names:
        out[k] = log_records[k]
    return out


def _summary_of(recs):
    """The TACO_EPISODE_SUMMARY_WORDS layout summed in float64 over records."""
    v = np.zeros(15)
    for t in range(3):
        r = recs[recs["task"] == t]
        ret = r["ret"].astype(np.float64)
        v[5 * t:5 * t + 5] = [len(r), (r["timed_out"] != 0).sum(), r["length"].astype(np.float64).sum(), ret.sum(), (ret * ret).sum()]
    return v


def _assert_summary_close(got, want, where):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    for t in range(3):
        a, b = got[5 * t:5 * t + 5], want[5 * t:5 * t + 5]
        assert np.array_equal(a[:3], b[:3]), f"{where}: task {t} counts {a[:3]} != {b[:3]}"
        for j in (3, 4):
            assert abs(a[j] - b[j]) <= 1e-12 * max(abs(b[j]), 1e-300), f"{where}: task {t} word {j}: {a[j]!r} vs {b[j]!r}"


def _env(task, n, seed, max_len=25, **kw):
    import taco_b200
    cfg = taco_b200.make_cfg(task, n, domain_randomization=True)
    cfg["env"]["maxEpisodeLength"] = max_len
    return taco_b200.FpvVecTask(cfg, "cuda:0", "cuda:0", -1, True, seed=seed, **kw)


def _buffer(env, H):
    import taco_b200
    return taco_b200.RolloutBuffer(env.num_envs, 26, env.len_obs, 26, env.len_states, 4, H, 1, 0.99, 0.95, "cuda:0")


def _ring_rollout(env, buf, eps, first):
    """One rollout of buf.horizon_len random-action steps into the ring, then the scan.  Returns (new records, summary)."""
    if first:
        env.attach_rollout(buf)
    else:
        env.rewind_rollout()
    before = eps.count
    for _ in range(buf.horizon_len):
        env.step_raw(env.random_actions(env.step_count))
    summ = eps.scan().cpu().numpy().copy()
    return eps.read()[before:], summ


@pytest.mark.parametrize("task", ["pos", "flip", "mix"])
def test_records_equal_the_episode_log_of_a_ring_free_twin_and_the_stats(task):
    import taco_b200
    n, H, rollouts = 512, 16, 5                                  # 80 steps, 25-step episodes: they cross rollout boundaries
    a, a2, b = _env(task, n, 7), _env(task, n, 7), _env(task, n, 7)
    buf, buf2 = _buffer(a, H), _buffer(a2, H)
    eps, eps2 = taco_b200.RolloutEpisodes(a, 100000), taco_b200.RolloutEpisodes(a2, 100000)
    log = taco_b200.EpisodeLog(b, 100000)
    a.stats()
    got, total = [], np.zeros(15)
    for r in range(rollouts):
        recs, summ = _ring_rollout(a, buf, eps, r == 0)
        _, summ2 = _ring_rollout(a2, buf2, eps2, r == 0)
        for _ in range(H):
            b.step_raw(b.random_actions(b.step_count))
        # 3. the summary is the float64 sum of the scan's records; the twin's scan of the same rows is bit-identical
        _assert_summary_close(summ, _summary_of(recs), f"rollout {r}")
        assert summ.tobytes() == summ2.tobytes(), f"rollout {r}: twin summaries differ"
        got.append(recs)
        total += summ
    got = _sorted(np.concatenate(got))
    assert eps.dropped == 0 and len(got) == eps.count > n
    assert got["timed_out"].any() and not got["timed_out"].all()
    assert (got["end_step"] % H < got["length"] - 1).any()          # some episodes started in an earlier rollout
    # 1. bit for bit the first six fields of the ring-free twin's episode-log records
    want = _sorted(_first_six(log.read()))
    assert got.tobytes() == want.tobytes()
    if task == "mix":
        assert set(np.unique(got["task"])) == {0, 1, 2}
    # 2. against taco_env_stats over the same steps
    s = a.stats().cpu().numpy()
    assert total[0::5].sum() == s[1] and total[1::5].sum() == s[2] and total[2::5].sum() == s[4]
    assert abs(total[3::5].sum() - s[3]) <= 1e-5 * abs(s[3])     # the stats round their warp sums in float32
    for x in (eps, eps2, log):
        x.close()
    for e in (a, a2, b):
        e.close()


class RowReplay:
    """The scan's definitions replayed on the host over the ring rows: float32 return in step order, length, live flag."""

    def __init__(self, gids, task, live):
        self.gids, self.task = np.asarray(gids, np.int64), np.asarray(task)
        n = len(self.gids)
        self.ret, self.len = np.zeros(n, f32), np.zeros(n, np.int64)
        self.live = np.asarray(live, bool).copy()
        self.records = []

    def restart(self, live):
        self.ret[:], self.len[:] = 0, 0
        self.live = np.asarray(live, bool).copy()

    def rows(self, buf, k0, k1, step0):
        rew = buf.rew_buf[k0:k1, :, 0].cpu().numpy()
        done = buf.done_buf[k0:k1, :, 0].cpu().numpy() != 0
        tout = buf.timeout_buf[k0:k1, :, 0].cpu().numpy()
        for k in range(k1 - k0):
            self.ret = (self.ret + rew[k]).astype(f32)
            self.len += 1
            for e in np.flatnonzero(done[k] & self.live):
                self.records.append((self.gids[e], step0 + k, self.len[e], self.task[e], int(tout[k, e] != 0), self.ret[e]))
            self.ret[done[k]], self.len[done[k]] = 0, 0
            self.live |= done[k]

    def result(self):
        return np.array(self.records, dtype=_rec_dtype())


def _tasks(env):
    gid = env.env_offset + np.arange(env.num_envs)
    n1, n2 = int(env.num_envs_global / 3 * 1), int(env.num_envs_global / 3 * 2)
    return np.where(gid < n1, 0, np.where(gid < n2, 1, 2))


def test_start_rule_attach_mid_run_reset_all_reattached_ring_and_rewind_with_unscanned_rows():
    import taco_b200
    n, H = 1024, 40
    env = _env("mix", n, 11, max_len=10)                         # time-outs end most episodes at steps 8, 17, 26, 35, ...
    buf = _buffer(env, H)
    reset_now = lambda: env.reset_buf.cpu().numpy() != 0

    def steps(k):
        for _ in range(k):
            env.step_raw(env.random_actions(env.step_count))

    env.attach_rollout(buf)
    steps(13)                                                    # rows 0..12 are written before the records are attached
    eps = taco_b200.RolloutEpisodes(env, 100000)
    replay = RowReplay(np.arange(n), _tasks(env), reset_now())
    assert not replay.live.all()                                 # mid-episode envs: their episode ending at step 17 is not recorded
    steps(H - 13)
    eps.scan()
    replay.rows(buf, 13, H, 13)
    checks = []

    def check(where):
        torch.cuda.synchronize()
        got, want = _sorted(eps.read()), _sorted(replay.result())
        assert len(got) > 0, where
        assert got.tobytes() == want.tobytes(), where
        checks.append(where)

    check("attach mid-run")
    # a rewind over unscanned rows restarts the rule: the rows are never scanned, the envs mid-episode are not recorded
    env.rewind_rollout()
    steps(9)
    env.rewind_rollout()
    replay.restart(reset_now())
    t0 = env.step_count
    steps(H)
    eps.scan()
    replay.rows(buf, 0, H, t0)
    check("rewind with unscanned rows")
    # steps without a ring are unseen: attaching the ring again restarts the rule
    env.detach_rollout()
    steps(5)
    env.attach_rollout(buf)
    replay.restart(reset_now())
    t0 = env.step_count
    steps(H)
    eps.scan()
    replay.rows(buf, 0, H, t0)
    check("re-attached ring")
    # reset_all: every env starts fresh, the episodes in progress are discarded
    env.rewind_rollout()
    steps(6)
    env.reset_all()
    replay.restart(np.ones(n, bool))
    steps(H)
    eps.scan()
    replay.rows(buf, 0, H, 0)
    check("reset_all")
    # a scan with no new rows appends nothing and reports an empty summary; a rewind after a scan keeps the episodes in progress
    count = eps.count
    assert not eps.scan().any() and eps.count == count
    env.rewind_rollout()
    t0 = env.step_count
    steps(H)
    eps.scan()
    replay.rows(buf, 0, H, t0)
    check("rewind after a scan")
    got = eps.read()
    # every record holds a whole episode: it started after the rule last ran for its env
    assert (got["length"] >= 1).all() and len(checks) == 5
    eps.close()
    env.close()


def test_capacity_drops_but_counts_and_the_summary_covers_every_episode():
    import taco_b200
    n, H, cap = 1024, 16, 300
    runs = []
    for capacity in (100000, cap):
        env = _env("pos", n, 5)
        buf = _buffer(env, H)
        eps = taco_b200.RolloutEpisodes(env, capacity)
        summ = [_ring_rollout(env, buf, eps, r == 0)[1] for r in range(3)]
        torch.cuda.synchronize()
        runs.append((eps.read().copy(), eps.count, eps.dropped, summ))
        eps.close()
        env.close()
    (full, n_full, d_full, s_full), (part, n_part, d_part, s_part) = runs
    assert d_full == 0 and n_full == len(full) > cap
    assert n_part == n_full and d_part == n_full - cap and len(part) == cap
    full_keys = {r.tobytes() for r in full}
    assert all(r.tobytes() in full_keys for r in part)
    # scans append in order (within a scan in an unspecified order): every record of the scans before the one that crossed the
    # capacity is kept, and none of a later scan
    crossed = int(np.searchsorted(np.cumsum([v[0::5].sum() for v in s_full]), cap, side="right"))
    part_keys = {r.tobytes() for r in part}
    assert all(r.tobytes() in part_keys for r in full[full["end_step"] < crossed * H])
    assert part["end_step"].max() < (crossed + 1) * H
    for a, b in zip(s_full, s_part):
        assert a.tobytes() == b.tobytes()


def test_invalid_calls():
    import taco_b200
    from taco_b200 import _capi
    lib = _capi.lib()
    n = 256
    env = _env("pos", n, 1)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    out = torch.zeros(15, dtype=torch.float64, device="cuda:0")
    scan = lambda: lib.taco_env_scan_rollout_episodes(env._h, C.c_void_p(out.data_ptr()), stream)
    assert scan() == _capi_invalid()                             # nothing attached
    assert lib.taco_env_rollout_episodes_clear(env._h, stream) == _capi_invalid()
    assert lib.taco_env_attach_rollout_episodes(env._h, 0, stream) == _capi_invalid()
    eps = taco_b200.RolloutEpisodes(env, 100)
    assert lib.taco_env_attach_rollout_episodes(env._h, 100, stream) == _capi_invalid()
    with pytest.raises(RuntimeError, match="no rollout ring"):   # no ring
        eps.scan()
    buf = _buffer(env, 4)
    p = lambda t: C.c_void_p(t.data_ptr())
    assert lib.taco_env_attach_rollout(env._h, p(buf.obs_ring), p(buf.states_ring), 5, None, None, None, stream) == 0
    env.step_raw(env.random_actions(0))
    assert scan() == _capi_invalid()                             # a ring without result rows
    assert lib.taco_env_scan_rollout_episodes(env._h, None, stream) == _capi_invalid()
    assert lib.taco_env_detach_rollout(env._h, stream) == 0
    # the episode log still refuses a ring, with or without rollout episodes
    env.attach_rollout(buf)
    with pytest.raises(RuntimeError, match="rollout ring"):
        taco_b200.EpisodeLog(env, 100)
    env.step_raw(env.random_actions(1))
    eps.scan()
    eps.close()
    assert scan() == _capi_invalid()                             # detached
    env.close()


def _capi_invalid():
    return -1                                                    # TACO_E_INVALID


def _graph_nets(gen):
    import taco_b200
    sizes = [26, 64, 64, 4]
    actor = taco_b200.ActorMLP(26, [64, 64], 4)
    actor.load([torch.randn(sizes[i + 1], sizes[i], generator=gen) * 0.25 for i in range(3)], [torch.zeros(sizes[i + 1]) for i in range(3)],
               log_std=torch.full((4,), -0.3))
    hid, mlp = 32, [64]
    lstm = [(torch.randn(4 * hid, 26, generator=gen) * 0.3, torch.randn(4 * hid, hid, generator=gen) * 0.2,
             torch.randn(4 * hid, generator=gen) * 0.1, torch.randn(4 * hid, generator=gen) * 0.1)]
    cs = [hid] + mlp + [1]
    critic = taco_b200.CriticLSTM(26, 5, hid, mlp)
    critic.load(lstm, [torch.randn(cs[i + 1], cs[i], generator=gen) / cs[i] ** 0.5 for i in range(2)],
                [torch.randn(cs[i + 1], generator=gen) * 0.1 for i in range(2)])
    return actor, critic


def test_graphed_rollout_records_and_summaries_equal_the_eager_loop():
    import taco_b200
    n, H, rollouts = 3000, 7, 4
    runs = {}
    for mode in ("eager", "graph", "graph_plain"):
        env = _env("mix", n, 21, max_len=9)
        actor, critic = _graph_nets(torch.Generator().manual_seed(2))
        buf = _buffer(env, H)
        eps = taco_b200.RolloutEpisodes(env, 100000) if mode != "graph_plain" else None
        gr, snaps = None, []
        for k in range(rollouts):
            before = eps.count if eps is not None else 0
            if mode == "eager":
                stats = taco_b200.collect_rollout(env, actor, buf, critic, seed=4, tensor_cores=True, episodes=eps)
            elif k == 0:
                gr = taco_b200.GraphedRollout(env, actor, buf, critic, seed=4, tensor_cores=True, episodes=eps)
                stats = gr.first_stats
            else:
                stats = gr.run()
            torch.cuda.synchronize()
            snap = [t.clone() for t in (stats, buf.adv_buf, buf.ret_buf, buf.obs_ring)]
            if eps is not None:
                snap += [_sorted(eps.read()[before:]), eps.summary_vec.clone()]
            snaps.append(snap)
        if gr is not None:
            gr.close()
        if eps is not None:
            eps.close()
        runs[mode] = snaps
        env.close(); actor.close(); critic.close()
    n_rec = 0
    for k in range(rollouts):
        e, g, plain = runs["eager"][k], runs["graph"][k], runs["graph_plain"][k]
        for j in range(4):                                       # the rollout itself is unchanged by the scan
            assert torch.equal(e[j], g[j]) and torch.equal(g[j], plain[j]), (k, j)
        assert e[4].tobytes() == g[4].tobytes(), f"rollout {k}: records differ"
        assert torch.equal(e[5], g[5]), f"rollout {k}: summaries differ"
        _assert_summary_close(g[5].cpu().numpy(), _summary_of(g[4]), f"rollout {k}")
        n_rec += len(g[4])
    assert n_rec > n


def test_two_shards_sum_to_the_single_env():
    import taco_b200
    n, H, rollouts = 1500, 12, 3
    envs = [_env("mix", n, 3, max_len=10)] + [_env("mix", n // 2, 3, max_len=10, env_offset=off, num_envs_global=n) for off in (0, n // 2)]
    bufs = [_buffer(e, H) for e in envs]
    eps = [taco_b200.RolloutEpisodes(e, 100000) for e in envs]
    for r in range(rollouts):
        out = [_ring_rollout(e, b, x, r == 0) for e, b, x in zip(envs, bufs, eps)]
        _assert_summary_close(out[1][1] + out[2][1], out[0][1], f"rollout {r}")
    whole = _sorted(eps[0].read())
    parts = _sorted(np.concatenate([eps[1].read(), eps[2].read()]))
    assert whole.tobytes() == parts.tobytes() and len(whole) > n
    for x in eps:
        x.close()
    for e in envs:
        e.close()

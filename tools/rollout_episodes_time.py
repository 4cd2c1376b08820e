#!/usr/bin/env python
"""Cost of the training-time episode records (DESIGN.md section 6f, taco_b200.RolloutEpisodes), one JSON line per measurement:

  * "scan": the scan alone over one rollout's rows (mix, domain randomisation, random actions) at 4096 envs x 64 steps and at
    2 Mi envs x 32 steps -- its kernel time (torch.profiler over a window of its own) and its bytes / time as a fraction of the
    device-to-device copy bandwidth measured in the same run.  The same rows are scanned again on every replay of a graph of
    [counter clear, scan], so the per-env planes keep advancing but every replay reads and appends the same amount;
  * "graphed_rollout": ms per GraphedRollout replay with and without ``episodes`` (mix, horizon 64, the example's default nets),
    at 4096 and 262 144 envs, windows of the two alternating;
  * the GPU name and power limit, read in the same run.

    python tools/rollout_episodes_time.py [--out profiles/rollout_episodes_time_b200.jsonl]
"""
import argparse
import json
import os
import statistics
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from eval_time import copy_bandwidth, gpu_info, kernel_ms, time_steps  # noqa: E402

# bytes the scan moves per env-step of rows: done read twice (pass 1 counts the records, pass 2 writes them), rew, the time-out
# byte (read only at an episode end, counted in full); per env once: ret / len / live read and written; 24 B per record
ROW_BYTES, PLANE_BYTES, RECORD_BYTES = 4 + 4 + 4 + 1, 2 * (4 + 4 + 1), 24


def scan_cost(torch, taco_b200, n, H, bw):
    env = taco_b200.FpvVecTask(taco_b200.make_cfg("mix", n, domain_randomization=True), "cuda:0", "cuda:0", -1, True, seed=1)
    buf = taco_b200.RolloutBuffer(n, 26, env.len_obs, 26, env.len_states, 4, H, 1, 0.99, 0.95, "cuda:0")
    eps = taco_b200.RolloutEpisodes(env, n * H)
    env.attach_rollout(buf)
    for _ in range(H):
        env.step_raw(env.random_actions(env.step_count))
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()                                   # the rows stay unscanned on the host: every replay rescans them
    with torch.cuda.graph(g):
        eps.clear()
        eps.scan()
    g.replay()
    torch.cuda.synchronize()
    records = eps.count
    reps = 50 if n >= 1 << 20 else 2000
    ms, launches = kernel_ms(torch, g.replay, reps, "rollout_episodes_scan")
    nbytes = ROW_BYTES * n * H + PLANE_BYTES * n + RECORD_BYTES * records
    out = {"measure": "scan", "task": "mix", "num_envs": n, "rows": H, "records_per_scan": records, "scan_kernel_ms": ms,
           "scan_launches_profiled": launches, "bytes_per_scan": nbytes, "bytes_per_s": nbytes / (ms * 1e-3),
           "fraction_of_copy_bw": nbytes / (ms * 1e-3) / bw, "replay_ms": statistics.median(time_steps(torch, g.replay, reps) for _ in range(3))}
    g = None
    eps.close()
    env.close()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    return out


def graphed_cost(torch, taco_b200, n, H=64):
    gen = torch.Generator().manual_seed(0)
    a_sizes, hid, c_mlp = [26, 256, 256, 256, 4], 64, [256, 256]
    aw = [torch.randn(a_sizes[i + 1], a_sizes[i], generator=gen) / a_sizes[i] ** 0.5 for i in range(4)]
    ab = [torch.zeros(a_sizes[i + 1]) for i in range(4)]
    lstm = [(torch.randn(4 * hid, 26, generator=gen) * 0.2, torch.randn(4 * hid, hid, generator=gen) * 0.1,
             torch.zeros(4 * hid), torch.zeros(4 * hid))]
    cs = [hid] + c_mlp + [1]
    cw = [torch.randn(cs[i + 1], cs[i], generator=gen) / cs[i] ** 0.5 for i in range(3)]
    cb = [torch.zeros(cs[i + 1]) for i in range(3)]
    runs = {}
    for mode in ("plain", "episodes"):
        env = taco_b200.FpvVecTask(taco_b200.make_cfg("mix", n, domain_randomization=True), "cuda:0", "cuda:0", -1, True, seed=1)
        actor = taco_b200.ActorMLP(26, a_sizes[1:-1], 4)
        actor.load(aw, ab)
        critic = taco_b200.CriticLSTM(26, env.len_states, hid, c_mlp)
        critic.load(lstm, cw, cb)
        buf = taco_b200.RolloutBuffer(n, 26, env.len_obs, 26, env.len_states, 4, H, 1, 0.99, 0.95, "cuda:0")
        eps = taco_b200.RolloutEpisodes(env, n) if mode == "episodes" else None
        tc = actor.tensor_cores_available and critic.tensor_cores_available
        gr = taco_b200.GraphedRollout(env, actor, buf, critic, seed=1, tensor_cores=tc, episodes=eps)
        for _ in range(3):
            gr.run()
        runs[mode] = (env, actor, critic, eps, gr, tc)
    reps = 5 if n >= 1 << 18 else 50
    t = {"plain": [], "episodes": []}
    for _ in range(5):                                           # alternating windows
        for mode in ("plain", "episodes"):
            t[mode].append(time_steps(torch, runs[mode][4].run, reps))
    out = {"measure": "graphed_rollout", "task": "mix", "num_envs": n, "horizon": H, "tensor_cores": bool(runs["plain"][5]),
           "replays_per_window": reps, "replay_ms": statistics.median(t["plain"]),
           "replay_ms_with_episodes": statistics.median(t["episodes"]),
           "windows_ms": t, "episodes_last_rollout": runs["episodes"][3].summary()}
    out["added_fraction"] = out["replay_ms_with_episodes"] / out["replay_ms"] - 1.0
    for env, actor, critic, eps, gr, _ in runs.values():
        gr.close()
        if eps is not None:
            eps.close()
        env.close(); actor.close(); critic.close()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scan", default="4096x64,2097152x32", help="envs x rows of the scan measurements")
    ap.add_argument("--graphed", default="4096,262144", help="env counts of the GraphedRollout measurements")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import taco_b200
    if not torch.cuda.is_available():
        raise SystemExit("rollout_episodes_time.py measures on the GPU; there is no CUDA device")
    info = gpu_info(torch)
    bw = copy_bandwidth(torch)
    lines = []
    for spec in args.scan.split(","):
        n, H = (int(x) for x in spec.split("x"))
        lines.append(dict(scan_cost(torch, taco_b200, n, H, bw), copy_bw_bytes_per_s=bw, **info))
        print(json.dumps(lines[-1]), flush=True)
    for n in (int(x) for x in args.graphed.split(",")):
        lines.append(dict(graphed_cost(torch, taco_b200, n), **info))
        print(json.dumps(lines[-1]), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            for r in lines:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()

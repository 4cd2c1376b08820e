#!/usr/bin/env python
"""Cost of the evaluation path (DESIGN.md section 6f): the episode log's update against the step it follows, at the bench's
workload (flip, 2 Mi envs) and at the reference's scale (flip, 4096 envs).  Per workload, one JSON line:

  * ms per step of the step alone, of step + log update (CUDA events over a window of steps, median of 3 windows), and of a full
    graph-replayed evaluation step (actor mean -> step -> log; 64 steps per graph, as evaluate_policy runs them);
  * the log update's own kernel time (torch.profiler, CUDA activity of every launch in a window of its own) and its bytes / time as
    a fraction of the device-to-device copy bandwidth measured in the same run;
  * the GPU name and power limit, read in the same run.

    python tools/eval_time.py [--envs 2097152,4096] [--out profiles/eval_time.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

# bytes the update moves per env-step: rew 4, reset_buf 8, progress 4, state planes S0-S3 64 (+ S4 16 on flip envs),
# two accumulator float4 planes read and written 64; records (48 B per finished episode) are negligible
LOG_BYTES = {"flip": 4 + 8 + 4 + 64 + 16 + 64, "pos": 4 + 8 + 4 + 64 + 64}


def gpu_info(torch):
    try:
        pl = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=power.limit", "--format=csv,noheader"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as exc:                     # the number is still reported, without its power limit
        pl = f"unavailable ({exc!r})"
    return {"gpu": torch.cuda.get_device_name(), "power_limit": pl}


def copy_bandwidth(torch, nbytes=4 << 30, reps=10):
    src = torch.empty(nbytes // 4, dtype=torch.float32, device="cuda")
    dst = torch.empty_like(src)
    src.fill_(1.0)
    dst.copy_(src)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    best = 0.0
    for _ in range(3):
        e0.record()
        for _ in range(reps):
            dst.copy_(src)
        e1.record()
        e1.synchronize()
        best = max(best, 2 * nbytes * reps / (e0.elapsed_time(e1) * 1e-3))
    del src, dst
    torch.cuda.empty_cache()
    return best


def time_steps(torch, fn, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / steps


def kernel_ms(torch, fn, steps, needle):
    from torch.profiler import profile, ProfilerActivity
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            fn()
        torch.cuda.synchronize()
    tot, cnt = 0.0, 0
    for ev in prof.key_averages():
        if needle in ev.key:
            t = getattr(ev, "device_time_total", None)
            tot += (t if t is not None else ev.cuda_time_total)
            cnt += ev.count
    return (tot / cnt * 1e-3 if cnt else float("nan")), cnt


def workload(torch, taco_b200, n, bw, task="flip"):
    steps = 200 if n >= 1 << 20 else 2000
    env = taco_b200.FpvVecTask(taco_b200.make_cfg(task, n), "cuda:0", "cuda:0", -1, True, seed=1)
    acts = env.random_actions(0)
    step = lambda: env.step_raw(acts)
    for _ in range(20):
        step()
    out = {"task": task, "num_envs": n, "steps_per_window": steps}
    out["step_ms"] = statistics.median(time_steps(torch, step, steps) for _ in range(3))
    log = taco_b200.EpisodeLog(env, 1 << 22)
    for _ in range(20):
        step()

    def windows():
        r = []
        for _ in range(3):
            log.clear()                          # the windows keep appending (and writing) records
            r.append(time_steps(torch, step, steps))
        return r
    out["step_log_ms"] = statistics.median(windows())
    out["log_added_fraction"] = out["step_log_ms"] / out["step_ms"] - 1.0
    log.clear()
    out["log_kernel_ms"], out["log_kernel_launches"] = kernel_ms(torch, step, steps, "episode_log_update")
    out["step_kernel_ms"], _ = kernel_ms(torch, step, steps, "fpv_step_kernel")
    out["log_bytes_per_env_step"] = LOG_BYTES[task]
    out["log_bytes_per_s"] = LOG_BYTES[task] * n / (out["log_kernel_ms"] * 1e-3)
    out["log_fraction_of_copy_bw"] = out["log_bytes_per_s"] / bw
    out["episodes_logged_in_profile_window"] = log.count

    # full evaluation step: actor mean (26 -> 256 x 3 -> 4, tcgen05) -> step -> log, 64 steps per CUDA graph replay
    actor = taco_b200.ActorMLP(26, [256, 256, 256], 4)
    gen = torch.Generator().manual_seed(0)
    sizes = [26, 256, 256, 256, 4]
    actor.load([torch.randn(sizes[i + 1], sizes[i], generator=gen) / sizes[i] ** 0.5 for i in range(4)],
               [torch.zeros(sizes[i + 1]) for i in range(4)])
    tc = actor.tensor_cores_available
    a = torch.zeros(n, 4, device="cuda:0")
    S = 64

    def chunk():
        for _ in range(S):
            actor.forward(env.obs_buf, tensor_cores=tc, out=a)
            env.step_raw(a)
    chunk()
    torch.cuda.synchronize()
    env.graph_begin()
    before = env.step_count
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        chunk()
        env.graph_advance(S)
    env.step_count = before
    reps = max(1, steps // S)
    g.replay()
    log.clear()
    out["eval_step_ms"] = statistics.median(time_steps(torch, g.replay, reps) / S for _ in range(3))
    out["actor_tensor_cores"] = bool(tc)
    g = None
    env.graph_end()
    log.close()
    actor.close()
    env.close()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", default="2097152,4096")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import taco_b200
    if not torch.cuda.is_available():
        raise SystemExit("eval_time.py measures on the GPU; there is no CUDA device")
    info = gpu_info(torch)
    bw = copy_bandwidth(torch)
    lines = []
    for n in (int(x) for x in args.envs.split(",")):
        r = dict(workload(torch, taco_b200, n, bw), copy_bw_bytes_per_s=bw, **info)
        print(json.dumps(r), flush=True)
        lines.append(r)
    if args.out:
        with open(args.out, "w") as f:
            for r in lines:
                f.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    main()

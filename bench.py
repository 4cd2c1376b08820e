#!/usr/bin/env python
"""bench.py -- env-steps/s of the fused FPV step (flip task) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Metric (BASELINE.json): env-steps/s, flip task, device-timed, max over ranks.  One "step" = one
VecTask.step over every env of the job (10 x 1 ms control sub-steps + observation history + reward
+ masked reset per env).  Envs shard independently over the GPUs (weak scaling: fixed envs per GPU,
global Philox env ids); the only collective is one NCCL all-reduce of the 8-double rollout
statistics vector at the end of the timed rollout.

Prints ONE JSON line on rank 0.  `value` = device-resident throughput through FpvVecTask.step;
`e2e` = the same step through the C ABI's host-buffer entry point (pinned-host actions H2D,
rew/reset/time_outs D2H, every step); `roofline` = HBM roofline of the step kernel using the
algorithmic bytes of SURVEY.md section 8(d); `sustained` = an internal 300-step window of the same workload with its own clock
samples (independent of --steps); `cpu_baseline` = the oracle port (the reference's torch modules' arithmetic + restated glue,
pinned to the reference's own classes by tests/golden/glue_*.npz) timed on this host's cores on a bounded sample of the SAME
workload; `policy_loop`, `config3_mix_actor`, `config4_rotate`, `config5_mix_dr` = the other BASELINE.json workloads.

--dump-outputs DIR writes what the last of the K timed steps returned (obs, states, rew, reset, time_outs at a fixed seeded sample
of envs, and the rollout statistics of the timed window) as DIR/*.npy.  Inputs depend only on the arguments (seeded env, Philox
actions), so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# stdout carries exactly ONE JSON line: whatever native libraries print to file descriptor 1 (NCCL writes its version banner
# there when NCCL_DEBUG is set) is sent to stderr, and emit() writes the line to the real stdout.
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())

ALGO_BYTES_NO_DR = 1493      # SURVEY.md section 8(d): 16 + 637 + 416 + 424 (len_obs=1, len_states=5, no per-env DR)
ALGO_BYTES_DR = 1549
TASK = "flip"
SEED = 0x7AC0
DUMP_MAX_ENVS = 65536        # --dump-outputs: 26 + 5 x 26 + 3 floats + an env id = 644 B per env, 42 MB at most


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=20)        # SURVEY.md section 8(d): 20 warm-up steps
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs-per-gpu", type=int, default=2 * 1024 * 1024)
    ap.add_argument("--task", default=TASK, choices=["pos", "rotate", "flip", "mix"])
    ap.add_argument("--dr", action="store_true", help="per-env domain randomisation (BASELINE config 5)")
    ap.add_argument("--fast-fp", action="store_true", help="time the FMA-contracted kernel build instead of the default strict (-fmad=false) one")
    ap.add_argument("--cpu-envs", type=int, default=262144, help="envs per step of the bounded CPU sample (a 4096-env step is dispatch-bound on the CPU)")
    ap.add_argument("--cpu-steps", type=int, default=6)
    ap.add_argument("--no-extra-configs", action="store_true", help="skip policy_loop / config4 / config5")
    ap.add_argument("--horizon", type=int, default=32, help="rollout horizon of the policy_loop point (SURVEY.md section 8d suggests 32)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-small", action="store_true")
    ap.add_argument("--no-numa", action="store_true", help="multi-GPU runs: do not pin each rank to its GPU's NUMA node (comparison runs)")
    ap.add_argument("--no-actor", action="store_true", help="skip the BASELINE config 3 point (mix task + actor MLP in the rollout loop)")
    ap.add_argument("--actor-envs", type=int, default=262144)
    ap.add_argument("--actor-hidden", default="256,256,256", help="actor hidden sizes (not pinned by the reference: the YAML is missing; our stated default)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned (rank 0's shard; a fixed seeded sample of at most "
                         f"{DUMP_MAX_ENVS} envs) as DIR/<name>.npy, float32 / float64, for comparing two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return args


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def mark(self):
        return time.time()

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self, t0, t1):
        sm, mx, pw, reasons = [], [], [], set()
        for ts, line in self.rows:
            if ts < t0 - 0.05 or ts > t1 + 0.15:
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:   # timed region shorter than the sampling period: fall back to every sample we have
            for ts, line in self.rows:
                f = [x.strip() for x in line.split(",")]
                try:
                    sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
                except Exception:
                    pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "power_w_max": max(pw), "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------ CPU baseline (oracle port)
def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def workload_config(task, dr, n, world):
    """The `config` object: identical in the GPU arm and in the --impl reference arm (what is measured, not how)."""
    return {"workload": f"{task} task fused env step (BASELINE configs[1] scaled to {n} envs/GPU so the working set exceeds L2), "
                        f"len_obs=1, len_states=5, delay_time=20, rotor_response_time=0.017, substeps=2, "
                        f"{'per-env DR on' if dr else 'no per-env DR'}, U(-1,1) Philox actions",
            "envs_per_gpu": n, "global_envs": world * n, "parallelism": f"env-sharded x{world}",
            "l2": "inputs larger than L2 (working set ~%.1f GB/GPU)" % (n * 1900 / 1e9)}


def cpu_baseline(task, n_envs, steps, warm=1, dr=False, threads=None):
    """The reference's CPU path for this hot path = its torch control/reward modules driven by the restated FpvBase glue (pinned to
    the reference's own env classes, tests/golden/glue_*.npz) + our rigid-body stand-in (oracle/)."""
    import torch
    from oracle.fpv_env import RefFpvEnv
    from oracle import philox as px
    from taco_b200.config import make_cfg
    import numpy as np
    threads = threads or (os.cpu_count() or 1)
    torch.set_num_threads(threads)
    cfg = make_cfg(task, n_envs, domain_randomization=dr)
    env = RefFpvEnv(cfg, seed=SEED)
    n_act = min(warm + steps, 4)
    acts = [torch.from_numpy(px.u01(px.draw(SEED, env.gid, t, 0, px.STREAM_ACTIONS)) * np.float32(2) - np.float32(1)) for t in range(n_act)]
    for t in range(warm):
        env.step(acts[t % n_act])
    t0 = time.perf_counter()
    for t in range(warm, warm + steps):
        env.step(acts[t % n_act])
    dt = time.perf_counter() - t0
    return {"value": n_envs * steps / dt, "unit": "env-steps/s", "cores": threads, "kind": "port", "cpu_model": cpu_model(),
            "sample": f"{task} task, {n_envs} envs x {steps} steps after {warm} warm-up, oracle port (torch CPU float32, {threads} threads, "
                      f"{cpu_model()}), {dt:.1f} s",
            "ms_per_step": dt / steps * 1e3}


def cpu_baseline_extras():
    """BASELINE.md section 3: config 1 (pos task, 4096 envs -- the reference's own scale, README.md:41) with 1 thread and with all
    threads; also the flip task at 4096 envs.  A 4096-env step is dispatch-bound on the CPU (~150 tiny torch ops per sub-step)."""
    out = {}
    for key, task, thr, steps in (("config1_pos_4096_all_threads", "pos", None, 20), ("config1_pos_4096_1_thread", "pos", 1, 10),
                                  ("flip_4096_all_threads", "flip", None, 20)):
        try:
            r = cpu_baseline(task, 4096, steps, 2, False, threads=thr)
            out[key] = {k: r[k] for k in ("value", "unit", "cores", "sample", "ms_per_step")}
        except Exception as exc:
            out[key] = {"error": repr(exc)}
    return out


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path (oracle port; the reference env class itself cannot run
    on a GPU box: IsaacGym/PhysX binaries are absent) on the SAME workload config as the GPU arm, each step a bounded sample of
    --cpu-envs envs of it.  Rank 0 only."""
    if rank != 0:
        return
    steps = max(1, min(args.steps, 20))
    warm = max(1, min(args.warmup, 2))
    cb = cpu_baseline(args.task, args.cpu_envs, steps, warm, args.dr)
    line = {
        "impl": "reference", "metric": "env-steps/s", "value": cb["value"], "unit": "env-steps/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": cb["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.task, args.dr, args.envs_per_gpu, world),
        "cpu_baseline": {k: cb[k] for k in ("value", "unit", "cores", "kind", "sample", "cpu_model")},
        "e2e": {"value": cb["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ------------------------------------------------------------------------------------------------ ours
def time_steps(env, actions, steps, torch, dist, world):
    """K consecutive steps bracketed by barrier + synchronize; CUDA events on the launching stream.  Returns (ms, rollout stats,
    what the last step returned: (obs_dict, rew, reset, extras), views of the env's buffers that the next step overwrites)."""
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    last = None
    for t in range(steps):
        last = env.step(actions[t % len(actions)])
    stats = env.stats()
    if world > 1:
        dist.all_reduce(stats)                       # the one collective of the path: 8 doubles per rollout
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if world > 1:
        tmax = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        ms = float(tmax.item())
        dist.barrier()
    return ms, stats, last


def dump_outputs(out_dir, last, stats, n, torch):
    """--dump-outputs: the last timed step's return values at a fixed, seeded sample of env indices (all envs when there are at most
    DUMP_MAX_ENVS), plus the rollout statistics of the timed window.  Called before the next step overwrites the buffers."""
    import numpy as np
    obs_dict, rew, reset, extras = last
    if n > DUMP_MAX_ENVS:
        idx = torch.randperm(n, generator=torch.Generator().manual_seed(SEED))[:DUMP_MAX_ENVS].sort().values
    else:
        idx = torch.arange(n)
    idx_dev = idx.to(rew.device)
    arrays = {"env_index": idx.double(),
              "obs": obs_dict["obs"][idx_dev].float(), "states": obs_dict["states"][idx_dev].float(),
              "rew": rew[idx_dev].float(), "reset": reset[idx_dev].float(), "time_outs": extras["time_outs"][idx_dev].float(),
              "rollout_stats": stats.double()}
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())
    return {"dir": os.path.abspath(out_dir), "envs": int(idx.numel()), "files": sorted(k + ".npy" for k in arrays),
            "note": "values returned by the last timed step at the envs listed in env_index.npy (rank 0's shard), "
                    "and the rollout statistics of the timed window"}


def _timed(torch, fn, iters, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def actor_rollout_point(torch, taco_b200, dev, n, hidden, strict_fp, peaks, iters=50):
    """BASELINE config 3: mix task, n envs, spectral-normalised actor MLP inference in the rollout loop
    (obs -> actor.act -> clipped action -> env.step), random-init policy (orthogonal, gains sqrt2 / 0.01,
    nets_asymmetry.py:41-55), weights projected once (lipschitz 4, ppo_asymmetry.py:398-404)."""
    sizes = [26] + list(hidden) + [4]
    gen = torch.Generator().manual_seed(SEED)
    ws, bs = [], []
    for l in range(len(sizes) - 1):
        w = torch.empty(sizes[l + 1], sizes[l])
        torch.nn.init.orthogonal_(w, gain=(2 ** 0.5 if l + 2 < len(sizes) else 0.01), generator=gen)
        ws.append(w)
        bs.append(torch.zeros(sizes[l + 1]))
    actor = taco_b200.ActorMLP(26, list(hidden), 4, device=dev)
    actor.load(ws, bs, lipschitz_const=4.0)
    env = taco_b200.FpvVecTask(taco_b200.make_cfg("mix", n), dev, dev, -1, True, seed=SEED, strict_fp=strict_fp)
    acts = [env.random_actions(t) for t in range(4)]
    for t in range(5):
        env.step(acts[t % 4])
    obs = env.obs_buf.clone()
    mean = torch.empty(n, 4, device=dev)
    tc = actor.tensor_cores_available
    ms_fp32 = _timed(torch, lambda: actor.forward(obs, tensor_cores=False, out=mean), max(iters // 5, 5))
    ms_tc = _timed(torch, lambda: actor.forward(obs, tensor_cores=True, out=mean), iters) if tc else None
    precision = None
    if tc:            # the bf16-operand kernel against the FP32 kernel (the reference computes in FP32) on this batch of real observations
        d = (actor.forward(obs, tensor_cores=True) - actor.forward(obs, tensor_cores=False)).abs()
        precision = {"max_abs_err": float(d.max()), "mean_abs_err": float(d.mean()), "action_range": [-1.0, 1.0],
                     "policy_std_at_init": 1.0, "note": "action mean of the tcgen05 (bf16 operands, fp32 accumulation) kernel minus the FP32 CUDA-core kernel "
                                                        "on the bench's observation batch; the sampled action adds N(0, std^2) noise with std = exp(2 log_std)"}
    k = [0]

    def env_only():
        env.step(acts[k[0] % 4]); k[0] += 1

    def loop():
        _, clipped, _, _ = actor.act(env.obs_buf, k[0], seed=SEED, tensor_cores=tc)
        env.step(clipped); k[0] += 1

    ms_env = _timed(torch, env_only, iters)
    ms_loop = _timed(torch, loop, iters)
    # ---- the critic of the reference's training command (README.md:60-66: LSTM encoder over the 5 x 26 state history + MLP) joins
    # the loop: agent.act = actor sample + critic value (nets_asymmetry.py:326-352), then env.step
    crit = None
    try:
        c_hid, c_mlp = 64, list(hidden)
        cs = [c_hid] + c_mlp + [1]
        lstm = []
        w_ih = torch.empty(4 * c_hid, 26); w_hh = torch.empty(4 * c_hid, c_hid)
        torch.nn.init.xavier_uniform_(w_ih, generator=gen); torch.nn.init.xavier_uniform_(w_hh, generator=gen)      # LSTMEncoder.para_init
        lstm.append((w_ih, w_hh, torch.zeros(4 * c_hid), torch.zeros(4 * c_hid)))
        cw, cb = [], []
        for l in range(len(cs) - 1):
            w = torch.empty(cs[l + 1], cs[l])
            torch.nn.init.orthogonal_(w, gain=(2 ** 0.5 if l + 2 < len(cs) else 0.01), generator=gen)
            cw.append(w); cb.append(torch.zeros(cs[l + 1]))
        critic = taco_b200.CriticLSTM(26, 5, c_hid, c_mlp, device=dev)
        critic.load(lstm, cw, cb)
        value = torch.empty(n, 1, device=dev)
        ctc = critic.tensor_cores_available
        ms_c_fp32 = _timed(torch, lambda: critic.forward(env.states_buf, tensor_cores=False, out=value), 3, warm=1)
        ms_c_tc = _timed(torch, lambda: critic.forward(env.states_buf, tensor_cores=True, out=value), iters) if ctc else None

        def loop_ac():
            _, clipped, _, _ = actor.act(env.obs_buf, k[0], seed=SEED, tensor_cores=tc)
            critic.forward(env.states_buf, tensor_cores=ctc, out=value)
            env.step(clipped); k[0] += 1

        ms_loop_ac = _timed(torch, loop_ac, iters)
        c_flops = 5 * 2.0 * (26 + c_hid) * 4 * c_hid + 2.0 * sum(cs[i] * cs[i + 1] for i in range(len(cs) - 1))
        crit = {"workload": f"critic = LSTM(26 -> {c_hid}) over the 5-frame state history + MLP {'x'.join(map(str, cs))} (sizes are OUR stated default: "
                            "the reference YAML is missing), agent.act = actor sample + critic value, then env.step, every step",
                "value": n / (ms_loop_ac * 1e-3), "unit": "env-steps/s", "ms_per_step": ms_loop_ac, "critic_fp32_ms": ms_c_fp32,
                "critic_tc_ms": ms_c_tc, "critic_flops_per_env": c_flops, "gpu_launches_per_step": 3}
        if ms_c_tc:
            ach = c_flops * n / (ms_c_tc * 1e-3) / 1e12
            peak = float(peaks.get("bf16_tflops", 1590.0))
            crit["critic_roofline"] = {"bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                                       "kernel": "critic_tc_kernel", "speedup_vs_fp32_kernel": ms_c_fp32 / ms_c_tc}
        critic.close()
    except Exception as exc:      # the config-3 line must not be lost to the (newer) critic point
        crit = {"error": repr(exc)}
    flops = 2.0 * sum(sizes[i] * sizes[i + 1] for i in range(len(sizes) - 1))        # per env, SURVEY.md section 8(d)
    out = {"workload": f"mix task, {n} envs, actor {'x'.join(map(str, sizes))} (hidden sizes are OUR stated default: the reference YAML is missing), "
                       "random-init policy, spectral projection c=4 once per update, act -> clip -> step every step",
           "value": n / (ms_loop * 1e-3), "unit": "env-steps/s", "ms_per_step": ms_loop, "env_step_ms": ms_env,
           "actor_fp32_ms": ms_fp32, "actor_tc_ms": ms_tc, "actor_flops_per_env": flops, "gpu_launches_per_step": 2,
           "actor_tc_precision": precision, "with_critic": crit}
    if ms_tc:
        ach = flops * n / (ms_tc * 1e-3) / 1e12
        peak = float(peaks.get("bf16_tflops", 1590.0))
        out["actor_roofline"] = {"bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
                                 "peak_source": "measured burst (MEASURED_PEAKS.json bf16_tflops)" if "bf16_tflops" in peaks else "fallback (B200_PROFILING.md)",
                                 "kernel": "actor_tc_kernel", "speedup_vs_fp32_kernel": ms_fp32 / ms_tc}
    env.close(); actor.close()
    return out


def small_rollout_point(torch, taco_b200, dev, task, hidden, strict_fp, n=4096, horizon=32, reps=5):
    """The rollout loop at the reference's own scale (README.md:41: 4096 envs): agent.act (actor sample + LSTM critic value) + env.step
    + zero-copy store + GAE, eager (collect_rollout) against one CUDA-graph replay per rollout (GraphedRollout, critic chain as a
    parallel branch).  Random-init networks of the bench's stated default sizes."""
    gen = torch.Generator().manual_seed(SEED)
    sizes = [26] + list(hidden) + [4]
    ws = [torch.randn(sizes[i + 1], sizes[i], generator=gen) / sizes[i] ** 0.5 for i in range(len(sizes) - 1)]
    bs = [torch.zeros(sizes[i + 1]) for i in range(len(sizes) - 1)]
    c_hid, cs = 64, [64] + list(hidden) + [1]
    lstm = [(torch.randn(4 * c_hid, 26, generator=gen) * 0.2, torch.randn(4 * c_hid, c_hid, generator=gen) * 0.15, torch.zeros(4 * c_hid), torch.zeros(4 * c_hid))]
    cw = [torch.randn(cs[i + 1], cs[i], generator=gen) / cs[i] ** 0.5 for i in range(len(cs) - 1)]
    cb = [torch.zeros(cs[i + 1]) for i in range(len(cs) - 1)]
    out = {"workload": f"{task}, {n} envs, horizon {horizon}: actor {'x'.join(map(str, sizes))} + critic LSTM 64 / MLP {'x'.join(map(str, cs))} in the loop, GAE at the end"}
    for mode in ("eager", "graph"):
        env = taco_b200.FpvVecTask(taco_b200.make_cfg(task, n), dev, dev, -1, True, seed=SEED, strict_fp=strict_fp)
        actor = taco_b200.ActorMLP(26, list(hidden), 4, device=dev); actor.load(ws, bs, lipschitz_const=-1.0)
        critic = taco_b200.CriticLSTM(26, 5, c_hid, list(hidden), device=dev); critic.load(lstm, cw, cb)
        buf = taco_b200.RolloutBuffer(n, 26, 1, 26, 5, 4, horizon, 1, 0.99, 0.95, dev)
        tc = actor.tensor_cores_available and critic.tensor_cores_available
        if mode == "eager":
            run = lambda: taco_b200.collect_rollout(env, actor, buf, critic, seed=SEED, tensor_cores=tc)
            run()
        else:
            gr = taco_b200.GraphedRollout(env, actor, buf, critic, seed=SEED, tensor_cores=tc)
            run = gr.run
        run()
        ms = _timed(torch, run, reps, warm=1)
        out[mode + "_ms_per_rollout"] = ms
        out[mode + "_env_steps_per_s"] = n * horizon / (ms * 1e-3)
        out[mode + "_us_per_step"] = ms / horizon * 1e3
        if mode == "graph":
            gr.close()
        env.close(); actor.close(); critic.close()
    return out


def kernel_source_sha():
    """sha256 (16 hex) of the step kernel's sources: ties profiles/traffic_bytes_per_env.json to the build under test."""
    import hashlib
    h = hashlib.sha256()
    for f in ("fpv_step_kernel.cuh", "fpv_math.cuh", "philox.cuh", "step_params.h"):
        with open(os.path.join(ROOT, "taco_b200", "csrc", f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()[:16]


def measured_traffic(task, dr):
    """(bytes per env-step from the committed ncu capture, note) -- only when the capture was taken from THIS kernel source."""
    tp = os.path.join(ROOT, "profiles", "traffic_bytes_per_env.json")
    if not os.path.exists(tp):
        return None, "no capture committed"
    try:
        t = json.load(open(tp))
    except Exception as exc:
        return None, repr(exc)
    key = task + ("_dr" if dr else "")
    if key not in t:
        return None, f"no capture for {key}"
    if t.get("kernel_source_sha16") != kernel_source_sha():
        return None, f"capture {t.get('capture', '?')} was taken from another kernel source ({t.get('kernel_source_sha16')}); re-run tools/gpu_traffic.sh"
    return float(t[key]), f"dram__bytes_read.sum + dram__bytes_write.sum per launch / envs, {t.get('capture', '?')}"


def shard_point(torch, dist, taco_b200, dev, rank, world, task, n, dr, strict_fp, peak, steps=100, warm=20):
    """One more BASELINE workload on this job's GPUs: fused step of `task` at n envs per GPU, weak-scaled, own HBM roofline."""
    cfg = taco_b200.make_cfg(task, n, domain_randomization=dr)
    env = taco_b200.FpvVecTask(cfg, dev, dev, -1, True, env_offset=rank * n, num_envs_global=world * n, seed=SEED, strict_fp=strict_fp)
    acts = [env.random_actions(t) for t in range(4)]
    for t in range(warm):
        env.step(acts[t % 4])
    env.stats()
    ms, _, _ = time_steps(env, acts, steps, torch, dist, world)
    env.close()
    algo = ALGO_BYTES_DR if dr else ALGO_BYTES_NO_DR
    ach = algo * n / (ms / steps * 1e-3) / 1e9
    return {"workload": f"{task} task, {n} envs/GPU x {world} GPUs = {world * n} envs{', per-env DR on' if dr else ''}, random actions, "
                        f"{steps} steps after {warm} warm-up, one stats all-reduce",
            "value": float(world) * n * steps / (ms * 1e-3), "unit": "env-steps/s", "ms_per_step": ms / steps, "n_gpus": world,
            "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "algorithmic_bytes_per_env_step": algo}}


def policy_loop_point(torch, dist, taco_b200, dev, rank, world, n, hidden, horizon, strict_fp, reps=5):
    """north_star "random-init-policy rollouts at 1, 2, 4, 8 GPUs": the whole collection loop of PPO.run on every rank's env shard
    -- horizon x (actor sample + LSTM critic value + env.step, zero-copy store), GAE, then the two small all-reduces (advantage
    moments, episode statistics) -- timed per rollout, max over ranks."""
    gen = torch.Generator().manual_seed(SEED)
    sizes = [26] + list(hidden) + [4]
    ws, bs = [], []
    for l in range(len(sizes) - 1):
        w = torch.empty(sizes[l + 1], sizes[l])
        torch.nn.init.orthogonal_(w, gain=(2 ** 0.5 if l + 2 < len(sizes) else 0.01), generator=gen)
        ws.append(w); bs.append(torch.zeros(sizes[l + 1]))
    c_hid, cs = 64, [64] + list(hidden) + [1]
    w_ih = torch.empty(4 * c_hid, 26); w_hh = torch.empty(4 * c_hid, c_hid)
    torch.nn.init.xavier_uniform_(w_ih, generator=gen); torch.nn.init.xavier_uniform_(w_hh, generator=gen)
    lstm = [(w_ih, w_hh, torch.zeros(4 * c_hid), torch.zeros(4 * c_hid))]
    cw, cb = [], []
    for l in range(len(cs) - 1):
        w = torch.empty(cs[l + 1], cs[l])
        torch.nn.init.orthogonal_(w, gain=(2 ** 0.5 if l + 2 < len(cs) else 0.01), generator=gen)
        cw.append(w); cb.append(torch.zeros(cs[l + 1]))
    env = taco_b200.FpvVecTask(taco_b200.make_cfg("mix", n), dev, dev, -1, True, env_offset=rank * n, num_envs_global=world * n,
                               seed=SEED, strict_fp=strict_fp)
    actor = taco_b200.ActorMLP(26, list(hidden), 4, device=dev); actor.load(ws, bs, lipschitz_const=4.0)
    critic = taco_b200.CriticLSTM(26, 5, c_hid, list(hidden), device=dev); critic.load(lstm, cw, cb)
    buf = taco_b200.RolloutBuffer(n, 26, 1, 26, 5, 4, horizon, 1, 0.99, 0.95, dev)
    run = lambda: taco_b200.collect_rollout(env, actor, buf, critic, seed=SEED, tensor_cores=True)
    run()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    # every rollout timed on its own and the MEDIAN reported: the loop is eager (101 launches per rollout), so one host hiccup
    # (a 90 ms stall of the launching thread was seen once in r02ak) would otherwise triple the mean of three; all values are in the line
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for e0, e1 in evs:
        e0.record()
        stats = run()
        e1.record()
    torch.cuda.synchronize()
    per_rollout = sorted(e0.elapsed_time(e1) for e0, e1 in evs)
    ms = per_rollout[len(per_rollout) // 2]
    if world > 1:
        tm = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
        ms = float(tm.item())
    env.close(); actor.close(); critic.close()
    return {"workload": f"mix task, {n} envs/GPU x {world} GPUs, horizon {horizon}: actor {'x'.join(map(str, sizes))} + critic LSTM 64 / MLP "
                        f"{'x'.join(map(str, cs))} (tcgen05 kernels; sizes are OUR stated default) + env.step every step, zero-copy store, GAE, "
                        "2 small all-reduces per rollout; random-init spectral-normalised policy",
            "value": float(world) * n * horizon / (ms * 1e-3), "unit": "env-steps/s", "ms_per_rollout": ms, "ms_per_step": ms / horizon,
            "ms_per_rollout_all": [round(x, 3) for x in per_rollout], "statistic": f"median of {reps} rollouts",
            "n_gpus": world, "gpu_launches_per_rollout": 3 * horizon + 5,
            "episodes_finished_last_rollout": float(stats[1].item())}


def native_update_point(torch, dev, hidden, n=4096, horizon=64, mb=4, iters=4, reps=3):
    """SURVEY.md section 8f row 4 at the reference's scale (README.md:41: 4096 envs): one PPO.update (ppo_asymmetry.py:137-258) =
    mb x iters optimiser steps on the rollout of n envs x horizon steps, on the native kernels (taco_ppo_*: tcgen05 GEMM forward /
    backward, device-side KL early stop, Adam, spectral projection) and on the PyTorch-autograd twin."""
    import types
    from taco_b200.ppo import PPOConfig, TorchActorCritic, make_optimizer, ppo_update
    from taco_b200.ppo_native import NativePPO
    agent = TorchActorCritic(26, 4, list(hidden), 26, 64, list(hidden)).to(dev)
    gen = torch.Generator(device=dev).manual_seed(SEED)
    rnd = lambda *sh: torch.randn(*sh, device=dev, generator=gen)
    buf = types.SimpleNamespace(obs_buf=rnd(horizon, n, 1, 26) * 0.5, states_buf=rnd(horizon, n, 5, 26) * 0.5, act_buf=rnd(horizon, n, 4).clamp(-1, 1),
                                value_buf=torch.zeros(horizon, n, 1, device=dev), ret_buf=rnd(horizon, n, 1) * 0.3, adv_buf=rnd(horizon, n, 1))
    with torch.no_grad():
        buf.logp_buf = agent.evaluate(buf.obs_buf.view(-1, 1, 26), buf.states_buf.view(-1, 5, 26), buf.act_buf.view(-1, 4))[0].view(horizon, n, 1)
    cfg = PPOConfig(train_iters=iters, use_lipschitz=True, lipschitz_para=4.0, target_kl=1e9)
    perm = torch.randperm(horizon * n, device=dev, generator=gen).view(mb, -1)
    idx = [perm[i] for i in range(mb)]
    nat = NativePPO(agent, perm.shape[1], device=dev)
    nat.update(buf, cfg, 0, batch_idx=idx)
    ms = _timed(torch, lambda: nat.update(buf, cfg, 1, batch_idx=idx), reps, warm=1)
    nat.close()
    opt = make_optimizer(agent, cfg)
    ppo_update(agent, opt, buf, cfg, 0, batch_idx=idx)
    ms_t = _timed(torch, lambda: ppo_update(agent, opt, buf, cfg, 1, batch_idx=idx), 1, warm=0)
    sizes = [26] + list(hidden) + [4]
    csz = [64] + list(hidden) + [1]
    flops = 3.0 * (2.0 * sum(sizes[i] * sizes[i + 1] for i in range(len(sizes) - 1)) + 5 * 2.0 * (26 + 64) * 256
                   + 2.0 * sum(csz[i] * csz[i + 1] for i in range(len(csz) - 1)))
    steps = mb * iters
    return {"workload": f"PPO.update on {n} envs x {horizon} steps: {mb} minibatches x {iters} iterations = {steps} optimiser steps of {perm.shape[1]} samples; "
                        f"actor {'-'.join(map(str, sizes))}, critic LSTM 64 + MLP {'-'.join(map(str, csz))}, spectral projection on (sizes are OUR stated default)",
            "native_update_ms": ms, "native_ms_per_optim_step": ms / steps, "autograd_update_ms": ms_t, "speedup_vs_autograd": ms_t / ms,
            "flops_per_sample_fwd_bwd": flops, "achieved_tflops": flops * perm.shape[1] * steps / (ms * 1e-3) / 1e12,
            "samples_per_s": perm.shape[1] * steps / (ms * 1e-3)}


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    import torch
    import torch.distributed as dist
    import taco_b200
    from taco_b200 import _capi
    from taco_b200 import dist as tdist
    numa_cpus = tdist.bind_to_gpu_numa(local_rank) if (world > 1 and not args.no_numa) else None    # pinned host buffers next to the rank's GPU
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback for the product path)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    n = args.envs_per_gpu
    warmup = max(args.warmup, 3)
    strict = not args.fast_fp
    hidden = [int(x) for x in args.actor_hidden.split(",")]
    cfg = taco_b200.make_cfg(args.task, n, domain_randomization=args.dr)
    dev = f"cuda:{local_rank}"
    env = taco_b200.FpvVecTask(cfg, dev, dev, -1, True, env_offset=rank * n, num_envs_global=world * n, seed=SEED, strict_fp=strict)
    n_act = 4
    actions = [env.random_actions(t) for t in range(n_act)]     # synthetic U(-1,1), resident in HBM before timing
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for t in range(warmup):
        env.step(actions[t % n_act])
    warm_stats = env.stats()
    if world > 1:
        dist.all_reduce(warm_stats)                  # NCCL communicator set-up happens here, outside the timed region
    launches0 = _capi.launch_count()
    t0 = sampler.mark()
    ms, stats, last = time_steps(env, actions, args.steps, torch, dist, world)
    t1 = sampler.mark()
    dumped = dump_outputs(args.dump_outputs, last, stats, n, torch) if (args.dump_outputs and rank == 0) else None
    launches = _capi.launch_count() - launches0      # counted by the library: one per kernel it launched in the timed region
    if world > 1:
        lt = torch.tensor([launches], dtype=torch.float64, device="cuda")
        dist.all_reduce(lt)
        launches = int(lt.item())
    total_env_steps = float(world) * n * args.steps
    value = total_env_steps / (ms * 1e-3)
    # ---- sustained window: 300 more steps of the same workload (episodes desynchronised by now), own clock samples
    s0 = sampler.mark()
    ms_sus, _, _ = time_steps(env, actions, 300, torch, dist, world)
    s1 = sampler.mark()
    # ---- end-to-end through the host-buffer C-ABI call
    e2e = None
    if not args.no_e2e:
        k_e2e = min(args.steps, 20)
        h_act = [actions[t % n_act].cpu().pin_memory() for t in range(n_act)]
        h_rew = torch.empty(n, dtype=torch.float32).pin_memory()
        h_reset = torch.empty(n, dtype=torch.int64).pin_memory()
        h_tout = torch.empty(n, dtype=torch.uint8).pin_memory()
        h_flags = torch.empty(n, dtype=torch.uint8).pin_memory()

        def time_host_steps(k, fn):
            for t in range(2):
                fn(t)
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for t in range(k):
                fn(t)
            e1.record()
            torch.cuda.synchronize()
            ms_ = e0.elapsed_time(e1)
            if world > 1:
                tm = torch.tensor([ms_], dtype=torch.float64, device="cuda")
                dist.all_reduce(tm, op=dist.ReduceOp.MAX)
                ms_ = float(tm.item())
            return float(world) * n * k / (ms_ * 1e-3)

        ref_fmt = lambda t: env.step_host(h_act[t % n_act], h_rew, h_reset, h_tout)
        os.environ["TACO_HOST_MODE"] = "copy"          # the chunked copy pipeline (what pageable buffers get), for comparison
        v_copy = time_host_steps(min(k_e2e, 10), ref_fmt)
        os.environ["TACO_HOST_MODE"] = "mapped"        # default: the kernel reads / writes the pinned host buffers itself
        v_map = time_host_steps(k_e2e, ref_fmt)
        v_compact = time_host_steps(k_e2e, lambda t: env.step_host_compact(h_act[t % n_act], h_rew, h_flags))
        # e2e_full: obs and states cross PCIe too (they stay device-resident by design: the policy lives on the device)
        h_obs = torch.empty(n, 1, 26, dtype=torch.float32).pin_memory()
        h_states = torch.empty(n, 5, 26, dtype=torch.float32).pin_memory()

        def full(t):
            env.step_host(h_act[t % n_act], h_rew, h_reset, h_tout)
            h_obs.copy_(env.obs_buf, non_blocking=True); h_states.copy_(env.states_buf, non_blocking=True)
            torch.cuda.current_stream().synchronize()
        v_full = time_host_steps(min(k_e2e, 5), full)
        pcie_gbs = v_map / world * 29 / 1e9
        e2e = {"value": v_map, "unit": "env-steps/s", "steps": k_e2e,
               "h2d_bytes_per_step": n * 16, "d2h_bytes_per_step": n * 13, "copy_pipeline_value": v_copy,
               "compact": {"value": v_compact, "unit": "env-steps/s", "h2d_bytes_per_step": n * 16, "d2h_bytes_per_step": n * 5,
                           "note": "taco_env_step_host_compact: rew f32 + one flag byte (reset | time_out << 1) instead of f32 + int64 + bool"},
               "e2e_full": {"value": v_full, "unit": "env-steps/s", "h2d_bytes_per_step": n * 16, "d2h_bytes_per_step": n * (13 + 104 + 520),
                            "note": "additionally copies obs (104 B/env) and states (520 B/env) to pinned host memory every step"},
               "host_link": {"bytes_per_env": 29, "achieved_gb_per_s_per_gpu": pcie_gbs,
                             "note": "16 B in + 13 B out per env through one PCIe link per GPU; tools/probes/pcie_sm_probe.cu moves the same "
                                     "bytes with no arithmetic at the same rate (profiles/pcie_sm_probe_r01e.txt): the call is bound by "
                                     "the host link, and on this VM all GPUs share one host fabric (NUMA 0)"},
               "note": "per GPU bytes; taco_env_step_host with pinned host buffers, every step: one launch whose threads load their "
                       "action from host memory and post rew/reset/time_outs into host memory across PCIe, then a stream sync; "
                       "copy_pipeline_value = the same call with TACO_HOST_MODE=copy (chunked cudaMemcpyAsync pipeline). "
                       "obs (104 B/env) and states (520 B/env) stay device-resident BY DESIGN -- the policy and the rollout buffer live on "
                       "the device (taco_actor_act / taco_env_attach_rollout read them in place); e2e_full is the same call with both "
                       "also copied to the host"}
    sampler.stop()
    clocks = sampler.summary(t0, t1) if rank == 0 else None
    clocks_sus = sampler.summary(s0, s1) if rank == 0 else None
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peaks = json.load(open(peaks_path)) if os.path.exists(peaks_path) else {}
    if "hbm_gbs" in peaks:
        peak, peak_src = float(peaks["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    # ---- small-N point of BASELINE config 2 (4096 envs, launch-latency bound)
    small = None
    if not args.no_small and world == 1:
        cfg_s = taco_b200.make_cfg(args.task, 4096)
        env_s = taco_b200.FpvVecTask(cfg_s, dev, dev, -1, True, seed=SEED, strict_fp=strict)
        acts_s = [env_s.random_actions(t) for t in range(n_act)]
        for t in range(10):
            env_s.step(acts_s[t % n_act])
        ms_s, _, _ = time_steps(env_s, acts_s, 200, torch, dist, 1)
        small = {"workload": f"{args.task}, 4096 envs (BASELINE config 2, the reference's own scale), L2-resident; bound by instruction latency, not by bandwidth",
                 "value": 4096 * 200 / (ms_s * 1e-3), "unit": "env-steps/s", "us_per_step": ms_s / 200 * 1e3}
        env_s.close()
        if not args.no_actor:
            try:
                small["rollout_loop"] = small_rollout_point(torch, taco_b200, dev, args.task, hidden, strict)
            except Exception as exc:
                small["rollout_loop"] = {"error": repr(exc)}
    env.close()
    extra = {}
    if not args.no_extra_configs and not args.no_actor:
        for key, fn in (("policy_loop", lambda: policy_loop_point(torch, dist, taco_b200, dev, rank, world, args.actor_envs, hidden, args.horizon, strict)),
                        ("config4_rotate", lambda: shard_point(torch, dist, taco_b200, dev, rank, world, "rotate", 524288, False, strict, peak)),
                        ("config5_mix_dr", lambda: shard_point(torch, dist, taco_b200, dev, rank, world, "mix", 2097152, True, strict, peak))):
            try:
                extra[key] = fn()
            except Exception as exc:      # all ranks take the same path: a failure here is deterministic, not rank-local
                extra[key] = {"error": repr(exc)}
        if "value" in extra.get("config4_rotate", {}):
            extra["config4_rotate"]["baseline_config"] = "BASELINE configs[3]: circle task, 4 Mi envs over 8 GPUs (exact at n_gpus = 8)"
        if "value" in extra.get("config5_mix_dr", {}):
            extra["config5_mix_dr"]["baseline_config"] = "BASELINE configs[4]: mix task, 16 Mi envs over 8 GPUs, per-env DR (exact at n_gpus = 8)"
    actor_pt = None
    if not args.no_actor and world == 1:
        actor_pt = actor_rollout_point(torch, taco_b200, dev, args.actor_envs, hidden, strict, peaks)
        try:
            extra["ppo_update_4096x64"] = native_update_point(torch, dev, hidden)
        except Exception as exc:
            extra["ppo_update_4096x64"] = {"error": repr(exc)}
    if rank == 0:
        algo = ALGO_BYTES_DR if args.dr else ALGO_BYTES_NO_DR
        kernel_ms = ms / args.steps
        achieved = algo * n / (kernel_ms * 1e-3) / 1e9
        tr_per_env, tr_note = measured_traffic(args.task, args.dr)
        ach_sus = algo * n / (ms_sus / 300 * 1e-3) / 1e9
        line = {
            "metric": "env-steps/s", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": args.steps, "warmup": warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": workload_config(args.task, args.dr, n, world),
            "fp_mode": "fast (FMA contraction)" if args.fast_fp else "strict (-fmad=false, the parity-tested build)",
            "rank0_numa_bound_cpus": (len(numa_cpus) if numa_cpus else None),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": (tr_per_env * n if tr_per_env is not None else None), "traffic_note": tr_note,
                         "kernel": "fpv_step_kernel", "algorithmic_bytes_per_env_step": algo, "peak_source": peak_src,
                         "kernel_ms": kernel_ms, "kernel_source_sha16": kernel_source_sha()},
            "sustained": {"steps": 300, "ms_per_step": ms_sus / 300, "value": float(world) * n * 300 / (ms_sus * 1e-3), "unit": "env-steps/s",
                          "roofline": {"bound": "hbm", "achieved": ach_sus, "peak": peak, "unit": "GB/s", "frac": ach_sus / peak},
                          "clocks": clocks_sus,
                          "note": "300 consecutive steps right after the timed region (episodes desynchronised, GPU at its sustained clocks)"},
            "gpu_launches": launches,
            "gpu_launches_note": "counted by the library (taco_launch_count) over the timed region, summed over ranks: one fused step kernel per step + the stats reduction",
            "clocks": clocks,
            "rollout_stats": [float(x) for x in stats.cpu().tolist()],
        }
        if dumped is not None:
            line["dump_outputs"] = dumped
        if e2e is not None:
            line["e2e"] = e2e
        if small is not None:
            line["config2_4096_envs"] = small
        if actor_pt is not None:
            line["config3_mix_actor"] = actor_pt
        line.update(extra)
        if not args.no_cpu_baseline and world == 1:
            cb = cpu_baseline(args.task, args.cpu_envs, args.cpu_steps, 1, args.dr)
            line["cpu_baseline"] = {k: v for k, v in cb.items() if k != "ms_per_step"}
            line["cpu_baseline"]["same_workload_gpu_value"] = value
            line["cpu_baseline_extra"] = cpu_baseline_extras()
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()

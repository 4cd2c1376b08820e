"""Host-side multi-GPU plumbing of the env-sharded rollout (SURVEY.md section 8e).

Envs are independent, so the path shards with no data-path collective: rank r of W simulates the global envs
[r*n, (r+1)*n).  Global ids key the Philox streams and the mix-task groups (fpv_asymmetry.py:924-926), so a shard
reproduces exactly the trajectories those envs have in a single-GPU run.  The one exchange is a SUM all-reduce of the
8-double rollout statistics vector (taco_env_stats), once per rollout -- the distributed form of the single-device
reductions at ppo_asymmetry.py:313-339 and buffer_asymmetry.py:132.  Works with NCCL (CUDA tensors) and gloo (CPU).
"""
import torch
import torch.distributed as dist

STAT_NAMES = ("sum_reward", "n_done", "n_timeout", "sum_episode_return", "sum_episode_length", "n_nonfinite",
              "n_delay_overflow", "n_env_steps")


def shard(rank, world_size, envs_per_rank):
    """-> (env_offset, num_envs_global) for FpvVecTask(env_offset=..., num_envs_global=...)."""
    if not (0 <= rank < world_size):
        raise ValueError(f"rank {rank} outside world of {world_size}")
    return rank * envs_per_rank, world_size * envs_per_rank


def mix_groups(num_envs_global):
    """Boundaries [0, n1, n2, N] of the pos / rotate / flip thirds, evaluated like fpv_asymmetry.py:924-926."""
    return [0, int(num_envs_global / 3 * 1), int(num_envs_global / 3 * 2), int(num_envs_global)]


def allreduce_rollout_stats(stats, group=None):
    """In-place SUM over ranks of the (8,) float64 statistics vector; no-op without an initialised process group."""
    if stats.dtype != torch.float64 or stats.numel() != len(STAT_NAMES):
        raise ValueError("stats must be a float64 tensor of 8 elements")
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.SUM, group=group)
    return stats


def summarise(stats):
    """Global rollout scalars the trainer logs (ppo_asymmetry.py:428-436) from the reduced vector."""
    s = {k: float(v) for k, v in zip(STAT_NAMES, stats.tolist())}
    steps = max(s["n_env_steps"], 1.0)
    eps = max(s["n_done"], 1.0)
    return {"mean_reward": s["sum_reward"] / steps, "mean_episode_return": s["sum_episode_return"] / eps,
            "mean_episode_length": s["sum_episode_length"] / eps, "done_rate": s["n_done"] / steps,
            "timeout_fraction": s["n_timeout"] / eps, **s}


EPISODE_SUMMARY_FIELDS = ("episodes", "time_outs", "sum_length", "sum_ret", "sum_ret2")
TASK_NAMES = ("pos", "rotate", "flip")


def allreduce_episode_summary(summary, group=None):
    """In-place SUM over ranks of the (15,) float64 per-task episode summary of a rollout (taco_env_scan_rollout_episodes); no-op
    without an initialised process group."""
    if summary.dtype != torch.float64 or summary.numel() != len(TASK_NAMES) * len(EPISODE_SUMMARY_FIELDS):
        raise ValueError("summary must be a float64 tensor of 15 elements")
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(summary, op=dist.ReduceOp.SUM, group=group)
    return summary


def summarise_episode_summary(summary):
    """Per-task scalars from a (reduced) episode summary: one dict per task with episodes, keyed "pos" / "rotate" / "flip", holding
    the raw sums plus survival (time-outs / episodes), ret_mean, ret_std (population) and length_mean."""
    v = summary.tolist() if hasattr(summary, "tolist") else list(summary)
    out = {}
    for t, name in enumerate(TASK_NAMES):
        s = dict(zip(EPISODE_SUMMARY_FIELDS, v[5 * t:5 * t + 5]))
        n = s["episodes"]
        if n <= 0:
            continue
        mean = s["sum_ret"] / n
        s.update(survival=s["time_outs"] / n, ret_mean=mean, ret_std=max(s["sum_ret2"] / n - mean * mean, 0.0) ** 0.5,
                 length_mean=s["sum_length"] / n)
        out[name] = s
    return out


def bind_to_gpu_numa(gpu_index):
    """Pin the calling process to the CPUs NVML reports as local to GPU ``gpu_index`` (its NUMA node), so that pinned host
    buffers allocated afterwards -- the action / result buffers of ``step_host`` -- live in memory next to that GPU's PCIe root
    port instead of on whichever socket torchrun happened to start the rank.  Returns the CPU set, or None when NVML or the
    affinity call is unavailable (nothing is changed then)."""
    import os
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
        ids = [v.strip() for v in vis.split(",") if v.strip()]
        if ids:                                              # CUDA index -> NVML index (or UUID) through the visibility list
            ident = ids[int(gpu_index)]
            handle = pynvml.nvmlDeviceGetHandleByIndex(int(ident)) if ident.isdigit() else pynvml.nvmlDeviceGetHandleByUUID(ident)
        else:
            handle = pynvml.nvmlDeviceGetHandleByIndex(int(gpu_index))
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(handle, words)
        cpus = {64 * w + b for w, m in enumerate(mask) for b in range(64) if (m >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return cpus
    except Exception:
        return None

"""Test-mode evaluation of a trained policy on the device: per-episode outcome records and trajectory recording.

The reference evaluates with ``--train_mode=testmodel`` (train_fpv_asymmetry_ppo.py:328-356): the deterministic policy (the action
mean, ``agent(obs)``) drives the env with ``maxEpisodeLength = 1000``, and its ``Logger`` (CTRL/logger.py) records env 0 one
episode at a time.  Here:

  * ``EpisodeLog(env, capacity)``: the env's episode log (``taco_env_attach_episode_log``).  Every step is followed by one launch
    that appends a ``TacoEpisode`` record per finished episode -- return, length, task, time-out, position error, tilt, speed,
    angular velocity, roll travel -- so that 10^5 - 10^6 episodes of a domain-randomised policy can be measured in one run;
  * ``evaluate_policy``: the deterministic rollout loop (actor mean -> step -> log [-> recorder]), replayed as a CUDA graph;
  * ``summarise_episodes``: per-task distribution summaries of the records (host only);
  * ``save_trajectories``: the recorded rows (``taco_env_record_state``: the 64-word ``export_state`` row + the 4 applied actions)
    split into one ``.npy`` (named fields) and one ``.csv`` per (env, episode).  Our own file format, not the reference's.
"""
import ctypes as C
import math
import os
import warnings

import numpy as np
import torch

from . import _capi

EPISODE_DTYPE = _capi.EPISODE_DTYPE
TASK_NAMES = {0: "pos", 1: "rotate", 2: "flip"}

# names of the taco_env_export_state words (DESIGN.md "state export"), then the 4 actions the step applied
STATE_COLUMNS = (["pos_x", "pos_y", "pos_z", "quat_x", "quat_y", "quat_z", "quat_w", "linvel_x", "linvel_y", "linvel_z",
                  "angvel_x", "angvel_y", "angvel_z", "target_pos_x", "target_pos_y", "target_pos_z",
                  "target_quat_x", "target_quat_y", "target_quat_z", "target_quat_w", "roll_old", "roll_continuous",
                  "rotor_speed_0", "rotor_speed_1", "rotor_speed_2", "rotor_speed_3", "pid_prev_err_x", "pid_prev_err_y",
                  "pid_prev_err_z", "command", "battery_u1", "battery_ec", "battery_time", "episode_return", "progress",
                  "delay_len", "queue_runs", "delay_overflow", "reset", "reserved_39"]
                 + [f"omega_poly_{j}" for j in range(5)] + ["aero_k_f", "aero_k_tau", "aero_d_x", "aero_d_y", "aero_k_th"]
                 + [f"lag_gain_{j}" for j in range(4)] + [f"reserved_{j}" for j in range(54, 64)])
TRAJ_COLUMNS = STATE_COLUMNS + [f"action_{j}" for j in range(_capi.NUM_ACTS)]
assert len(STATE_COLUMNS) == _capi.STATE_WORDS
_PROGRESS, _RESET = STATE_COLUMNS.index("progress"), STATE_COLUMNS.index("reset")


class EpisodeLog:
    """The env's episode log: ``capacity`` records on the device, appended by one launch after every step of ``env`` (also inside
    CUDA graphs).  Only whole episodes are recorded (an env that is mid-episode at attach is recorded from its next episode on);
    the record order is unspecified.  ``env.reset_all()`` / ``import_state`` / ``load_state_checkpoint`` discard the episodes in
    progress.  Not allowed while a rollout ring is attached."""

    def __init__(self, env, capacity):
        self.env = env
        self._lib = _capi.lib()
        _capi.check(self._lib.taco_env_attach_episode_log(env._h, int(capacity), self._stream()), "taco_env_attach_episode_log")
        rec, cnt, cap = C.c_void_p(), C.c_void_p(), C.c_int64()
        _capi.check(self._lib.taco_env_episode_log_buffers(env._h, C.byref(rec), C.byref(cnt), C.byref(cap)), "taco_env_episode_log_buffers")
        self.capacity = int(cap.value)
        self._count = _capi.wrap(cnt.value, (1,), "<i8", env.device, self)
        self._records = _capi.wrap(rec.value, (self.capacity * EPISODE_DTYPE.itemsize,), "|u1", env.device, self)
        self._open = True

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.env.device_id).cuda_stream)

    @property
    def count(self):
        """Records appended since attach / the last ``clear`` (dropped ones included).  Synchronises."""
        return int(self._count.item())

    @property
    def dropped(self):
        return max(0, self.count - self.capacity)

    def read(self):
        """The records as a numpy structured array (``EPISODE_DTYPE``): the count first, then one copy of that many records."""
        n = min(self.count, self.capacity)
        raw = self._records[:n * EPISODE_DTYPE.itemsize].cpu().numpy()
        return raw.view(EPISODE_DTYPE)

    def clear(self):
        """Rewind the counter; the episodes in progress continue."""
        _capi.check(self._lib.taco_env_episode_log_clear(self.env._h, self._stream()), "taco_env_episode_log_clear")

    def close(self):
        if self._open:
            self._open = False
            self._records = self._count = None
            _capi.check(self._lib.taco_env_detach_episode_log(self.env._h), "taco_env_detach_episode_log")

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def summarise_episodes(records):
    """One summary dict per task present in ``records`` (keys "pos" / "rotate" / "flip"): episodes, survival (the time-out
    fraction), return mean and 5th / 50th / 95th percentiles, mean length, mean of ``pos_err_mean``, 95th percentile of
    ``tilt_max``, means of ``speed_mean`` and ``angvel_max``; flip also ``flips_per_episode`` (mean of roll_travel / 2 pi)."""
    out = {}
    if len(records) == 0:
        return out
    for t in sorted(int(v) for v in np.unique(records["task"])):
        r = records[records["task"] == t]
        ret = r["ret"].astype(np.float64)
        s = {"task": TASK_NAMES.get(t, str(t)), "episodes": int(len(r)),
             "survival": float(np.mean(r["timed_out"] != 0)),
             "ret_mean": float(ret.mean()), "ret_p5": float(np.percentile(ret, 5)), "ret_p50": float(np.percentile(ret, 50)),
             "ret_p95": float(np.percentile(ret, 95)), "length_mean": float(r["length"].astype(np.float64).mean()),
             "pos_err_mean": float(r["pos_err_mean"].astype(np.float64).mean()),
             "tilt_max_p95": float(np.percentile(r["tilt_max"].astype(np.float64), 95)),
             "speed_mean": float(r["speed_mean"].astype(np.float64).mean()),
             "angvel_max_mean": float(r["angvel_max"].astype(np.float64).mean())}
        if t == _capi.TASK["flip"]:
            s["flips_per_episode"] = float((r["roll_travel"].astype(np.float64) / (2.0 * math.pi)).mean())
        out[s["task"]] = s
    return out


def save_trajectories(traj, path):
    """Write the rows of ``traj`` (as ``evaluate_policy`` returns it) split at the episode boundaries: for every recorded env and
    episode ``env<global id>_ep<k>.npy`` (structured array: ``step`` + ``TRAJ_COLUMNS``) and ``.csv`` (same named columns).  An
    episode ends at a row whose ``reset`` word is set; a segment cut by the start or the end of the recording (first row's
    progress != 1, or last row not an end) gets the suffix ``_partial``.  Returns the written paths."""
    os.makedirs(path, exist_ok=True)
    data, steps, gids = np.asarray(traj["data"], np.float32), np.asarray(traj["step"]), np.asarray(traj["env_ids"])
    dtype = np.dtype([("step", "<u4")] + [(c, "<f4") for c in TRAJ_COLUMNS])
    written = []
    for j, gid in enumerate(gids):
        rows = data[:, j]
        ends = np.flatnonzero(rows[:, _RESET] != 0)
        bounds = [0] + [int(e) + 1 for e in ends if e + 1 < len(rows)] + [len(rows)]
        for k, (a, b) in enumerate(zip(bounds[:-1], bounds[1:])):
            seg = rows[a:b]
            partial = seg[0, _PROGRESS] != 1 or seg[-1, _RESET] == 0
            name = os.path.join(path, f"env{int(gid)}_ep{k:04d}" + ("_partial" if partial else ""))
            arr = np.empty(len(seg), dtype=dtype)
            arr["step"] = steps[a:b]
            for c, col in enumerate(TRAJ_COLUMNS):
                arr[col] = seg[:, c]
            np.save(name + ".npy", arr, allow_pickle=False)
            with open(name + ".csv", "w") as f:
                f.write(",".join(["step"] + TRAJ_COLUMNS) + "\n")
                for st, row in zip(steps[a:b], seg):
                    f.write(str(int(st)) + "," + ",".join(repr(float(v)) for v in row) + "\n")
            written += [name + ".npy", name + ".csv"]
    return written


def evaluate_policy(env, actor, min_episodes, max_steps, tensor_cores=True, graph=True, record_env_ids=None, steps_per_replay=64,
                    capacity=None):
    """Deterministic test-mode rollouts: ``env.reset_all()``, then per step ``ActorMLP.forward`` (the action mean; its tanh bounds
    the actions to +-1 like the reference's ``agent(obs)``) -> ``env.step_raw`` -> the episode log's update [-> the recorder on
    ``record_env_ids`` (local ids) and the 4 applied actions next to its 64 words].  Steps run in chunks of ``steps_per_replay``;
    with ``graph=True`` the first chunk runs eagerly and the chunk is then captured once as a CUDA graph and replayed.  The host
    reads the record count once per chunk; the loop ends when ``min_episodes`` records are in or ``max_steps`` (rounded up to a
    whole chunk) are taken.  ``steps_per_replay`` must be even: without a rollout ring the observation history ping-pongs between
    two buffers every step, so only an even number of steps replays with the same addresses.

    The records are the episodes that ENDED inside the run: when ``min_episodes`` is not large against ``num_envs``, short
    episodes (crashes) are over-represented and no episode longer than the run is in -- to estimate survival, ask for several
    times ``num_envs`` episodes or set ``max_steps`` well beyond ``maxEpisodeLength``.

    ``capacity`` (records kept; default ``min_episodes + num_envs * steps_per_replay``, enough for any chunk) -- the dropped
    count is reported with a warning.  Returns (records, trajectories or None, ``summarise_episodes(records)``); trajectories =
    {"env_ids": global ids (k,), "local_ids": (k,), "step": step index of every row (T,), "data": (T, k, 68) float32}."""
    S = int(steps_per_replay)
    if S < 2 or S % 2:
        raise ValueError(f"steps_per_replay must be even and >= 2 (got {steps_per_replay}): the observation buffers ping-pong every step")
    if env.rollout_buffer is not None:
        raise ValueError("evaluate_policy: detach the rollout ring first (the episode log reads the env's own buffers)")
    N, dev = env.num_envs, env.device
    tc = bool(tensor_cores and actor.tensor_cores_available)
    if tensor_cores and not tc:
        from .rollout import _warn_fp32_fallback
        _warn_fp32_fallback(False, True)
    if capacity is None:
        capacity = int(min_episodes) + N * S
    ids = None
    if record_env_ids is not None:
        local = np.asarray(record_env_ids, dtype=np.int64).reshape(-1)
        if local.size == 0 or local.min() < 0 or local.max() >= N:
            raise ValueError(f"record_env_ids must be local env ids in [0, {N})")
        ids = torch.from_numpy(local.astype(np.int32)).to(dev)
        ids_long = ids.long()
        k = int(local.size)
        rec_states = torch.empty(S, k, _capi.STATE_WORDS, dtype=torch.float32, device=dev)
        rec_act = torch.empty(S, k, _capi.NUM_ACTS, dtype=torch.float32, device=dev)
    actions = torch.zeros(N, _capi.NUM_ACTS, dtype=torch.float32, device=dev)

    def chunk():
        for s in range(S):
            actor.forward(env.obs_buf, tensor_cores=tc, out=actions)
            env.step_raw(actions)
            if ids is not None:
                env.record_state(ids, out=rec_states[s])
                torch.index_select(actions, 0, ids_long, out=rec_act[s])

    env.reset_all()
    log = EpisodeLog(env, capacity)
    rows, steps_taken, g = [], 0, None
    try:
        while True:
            first = env.step_count
            if g is None:
                chunk()
            else:
                g.replay()
                env.step_count += S
            steps_taken += S
            if ids is not None:
                rows.append((np.arange(first, first + S, dtype=np.uint32),
                             torch.cat([rec_states, rec_act], dim=2).cpu().numpy()))
            if log.count >= min_episodes or steps_taken >= max_steps:
                break
            if graph and g is None:
                torch.cuda.synchronize(dev)
                env.graph_begin()
                before = env.step_count
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    chunk()
                    env.graph_advance(S)
                env.step_count = before                    # the capture advanced the host mirrors without running anything
        records = log.read()
        if log.dropped:
            warnings.warn(f"evaluate_policy: {log.dropped} episode records past the capacity of {log.capacity} were dropped",
                          RuntimeWarning, stacklevel=2)
    finally:
        if g is not None:
            g = None
            env.graph_end()
        log.close()
    traj = None
    if ids is not None:
        traj = {"env_ids": local + env.env_offset, "local_ids": local, "step": np.concatenate([r[0] for r in rows]),
                "data": np.concatenate([r[1] for r in rows], axis=0)}
    return records, traj, summarise_episodes(records)

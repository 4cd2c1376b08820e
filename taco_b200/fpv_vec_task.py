"""Drop-in ``VecTask`` for the TACO fpv_asymmetry tasks, backed by the fused sm_100a step kernel.

Mirrors the surface train_fpv_asymmetry_ppo.py / ppo_asymmetry.py consume (SURVEY.md section 8b):

  * constructor ``Task(cfg, rl_device, sim_device, graphics_device_id, headless,
    virtual_screen_capture, force_render)``          fpv_asymmetry.py:54, train_fpv_asymmetry_ppo.py:363-371
  * ``isaacgym_task_map["Fpv_pos|Fpv_rotate|Fpv_flip|Fpv_mix"]``   tasks/__init__.py:33-39
  * attributes num_envs, num_obs, num_states, num_acts, len_obs, len_states, observation_space,
    state_space, action_space, difficulty (read/write), obs_buf, states_buf, rew_buf, reset_buf,
    progress_buf                                      vec_task_asymmetry.py:82-100,231-254
  * ``reset() -> {"obs","states"}``                   vec_task_asymmetry.py:352-361
  * ``step(actions) -> (obs_dict, rew, reset, {"time_outs"})``   vec_task_asymmetry.py:290-334

Everything below ``step`` runs in one CUDA kernel behind the C ABI (include/taco_b200.h).  The
returned tensors are zero-copy views of library-owned device buffers and are overwritten by the
next ``step`` (the reference returns fresh clamp() results for obs/states and the persistent
rew_buf/reset_buf; its only consumer copies everything before stepping again,
ppo_asymmetry.py:321-329).  There is no CPU fallback: constructing the env without CUDA raises.
"""
import ctypes as C
import math

import numpy as np
import torch

from . import _capi


class Box:
    """Shape/bounds holder standing in for gym.spaces.Box (gym is not a dependency here);
    the trainer reads .shape, .low, .high (ppo_asymmetry.py:42-52)."""

    def __init__(self, low, high):
        self.low = np.asarray(low, dtype=np.float32)
        self.high = np.asarray(high, dtype=np.float32)
        self.shape = self.low.shape
        self.dtype = np.float32


def _device_index(sim_device):
    dev = torch.device(sim_device if sim_device is not None else "cuda:0")
    if dev.type != "cuda":
        raise RuntimeError(f"FpvVecTask runs on CUDA only (got sim_device={sim_device!r}); there is no CPU path")
    return dev.index if dev.index is not None else 0


class FpvVecTask:
    task_mode = None   # set by subclasses; falls back to cfg["task_mode"]

    def __init__(self, cfg, rl_device="cuda:0", sim_device="cuda:0", graphics_device_id=-1, headless=True,
                 virtual_screen_capture=False, force_render=False, *, env_offset=0, num_envs_global=None, seed=None,
                 strict_fp=True, debug_delay=False):
        # strict_fp=True (default): the -fmad=false kernel build, op-for-op float32 like eager torch -- the build
        # every parity claim is made for and the one bench.py times.  strict_fp=False selects the FMA-contracted build.
        if not torch.cuda.is_available():
            raise RuntimeError("CUDA is not available: the fused FPV step has no CPU fallback")
        self.cfg = cfg
        env_cfg = cfg["env"]
        mode = self.task_mode or cfg.get("task_mode")
        if mode not in _capi.TASK:
            raise ValueError(f"Invalid task_mode: {mode!r}")
        if cfg.get("physics_engine", "physx") not in ("physx", "flex"):      # vec_task_asymmetry.py:166-173
            raise ValueError(f"Invalid physics engine backend: {cfg['physics_engine']}")
        if cfg["sim"].get("up_axis", "z") not in ("z", "y"):                 # vec_task_asymmetry.py:423-426
            raise ValueError(f"Invalid physics up-axis: {cfg['sim']['up_axis']}")
        if int(cfg["delay_time_max"]) != 100:
            raise ValueError("delay_time_max must be 100 (hard-coded arange(100), fpv_asymmetry.py:329)")
        self.device_id = _device_index(sim_device)
        self.device = f"cuda:{self.device_id}"
        self.rl_device = rl_device
        self.headless = headless
        # fields the reference keeps (fpv_asymmetry.py:57-115, vec_task_asymmetry.py:82-100)
        self.max_episode_length = int(env_cfg["maxEpisodeLength"])
        self.debug_viz = env_cfg.get("enableDebugVis", False)
        self.randomization_params = cfg.get("task", {}).get("randomization_params", {})
        self.num_envs = int(env_cfg["numEnvs"])
        self.num_agents = env_cfg.get("numAgents", 1)
        self.num_acts = env_cfg["numActions"] = _capi.NUM_ACTS
        self.num_obs = env_cfg["numObservations"] = _capi.NUM_OBS
        self.num_states = env_cfg["numStates"] = _capi.NUM_OBS
        self.len_obs = int(env_cfg.get("lenObservations", 1))
        self.len_states = int(env_cfg.get("lenStates", self.len_obs))
        self.control_freq_inv = int(env_cfg.get("controlFrequencyInv", 1))
        self.clip_obs = float(env_cfg.get("clipObservations", np.inf))
        self.clip_states = float(env_cfg.get("clipStates", np.inf))
        self.clip_actions = float(env_cfg.get("clipActions", np.inf))
        self.substeps = int(cfg["sim"].get("substeps", 2))
        self.dt = float(np.float32(cfg["sim"]["dt"]))
        self.num_commands = 2
        self._difficulty = float(cfg["difficulty"])
        self.obs_space = Box(np.ones((self.len_obs, self.num_obs)) * -np.inf, np.ones((self.len_obs, self.num_obs)) * np.inf)
        self.state_space = Box(np.ones((self.len_states, self.num_states)) * -np.inf, np.ones((self.len_states, self.num_states)) * np.inf)
        self.act_space = Box(np.ones(self.num_acts) * -1.0, np.ones(self.num_acts) * 1.0)
        for key in _capi.FLAGS:
            if key not in cfg:
                raise KeyError(f"cfg is missing required key {key!r}")
        flags = sum(bit for key, bit in _capi.FLAGS.items() if cfg[key])
        if strict_fp:
            flags |= _capi.F_STRICT_FP
        if debug_delay:
            flags |= _capi.F_DEBUG_DELAY
        self.env_offset = int(env_offset)
        self.num_envs_global = int(num_envs_global) if num_envs_global is not None else self.num_envs
        self.seed = int(seed if seed is not None else cfg.get("seed", 0)) & 0xFFFFFFFFFFFFFFFF
        c = _capi.TacoCfg(
            abi_version=_capi.ABI_VERSION, num_envs=self.num_envs, env_offset=self.env_offset,
            num_envs_global=self.num_envs_global, task_mode=_capi.TASK[mode], len_obs=self.len_obs,
            len_states=self.len_states, max_episode_length=self.max_episode_length,
            control_freq_inv=self.control_freq_inv, substeps=self.substeps, delay_time=int(cfg["delay_time"]),
            flags=flags, dt=cfg["sim"]["dt"], rotor_response_time=cfg["rotor_response_time"],
            difficulty=self._difficulty, clip_actions=self.clip_actions, seed=self.seed)
        self._lib = _capi.lib()
        handle = C.c_void_p()
        _capi.check(self._lib.taco_env_create(C.byref(c), self.device_id, C.byref(handle)), "taco_env_create")
        self._h = handle
        self.rollout_buffer = None          # RolloutBuffer whose ring the step kernel writes into (attach_rollout)
        self._wrap_buffers()
        self.extras = {}
        self.obs_dict = {}
        self._actions_keepalive = None
        self._ring_cur = 0
        self.step_count = 0                 # RL steps since construction / reset_all = the Philox step index of the next step

    # ------------------------------------------------------------------ buffers
    def _wrap_buffers(self):
        b = _capi.TacoBuffers()
        _capi.check(self._lib.taco_env_buffers(self._h, C.byref(b)), "taco_env_buffers")
        N, dev = self.num_envs, self.device
        self._obs_ab = [_capi.wrap(b.obs_ab[k], (N, self.len_obs, self.num_obs), "<f4", dev, self) for k in range(2)]
        base, frames, period = C.c_void_p(), C.c_int32(), C.c_int32()
        _capi.check(self._lib.taco_env_states_strip(self._h, C.byref(base), C.byref(frames), C.byref(period)), "taco_env_states_strip")
        self._strip = _capi.wrap(base.value, (N, frames.value, self.num_states), "<f4", dev, self)
        self._strip_period = period.value
        self._ab_ptr = [int(b.obs_ab[0]), int(b.obs_ab[1])]
        self.rew_buf = _capi.wrap(b.rew, (N,), "<f4", dev, self)
        self.reset_buf = _capi.wrap(b.reset, (N,), "<i8", dev, self)
        self.timeout_buf = _capi.wrap(b.time_outs, (N,), "|b1", dev, self)
        self._progress_i32 = _capi.wrap(b.progress, (N,), "<i4", dev, self)
        if self.rollout_buffer is None:           # with a ring attached, obs points into the ring (reset_all keeps the ring)
            self._cur = self._ab_ptr.index(int(b.obs))

    @property
    def obs_buf(self):
        if self.rollout_buffer is not None:
            return self.rollout_buffer.obs_ring[self._ring_cur]
        return self._obs_ab[self._cur]

    @property
    def states_buf(self):
        """(num_envs, len_states, 26) state history.  Without a rollout ring attached: a strided view of the library's history strip
        (taco_env_states_strip), the window of the current step; the next period - len_states steps leave it intact."""
        if self.rollout_buffer is not None:
            return self.rollout_buffer.states_ring[self._ring_cur]
        p = self.step_count % self._strip_period
        return self._strip[:, p:p + self.len_states]

    @property
    def progress_buf(self):
        return self._progress_i32.long()       # reference dtype is int64 (vec_task_asymmetry.py:250-251)

    @property
    def observation_space(self):
        return self.obs_space

    @property
    def action_space(self):
        return self.act_space

    @property
    def num_actions(self):
        return self.num_acts

    @property
    def difficulty(self):
        return self._difficulty

    @difficulty.setter
    def difficulty(self, value):                 # written by the trainer every epoch (ppo_asymmetry.py:173-175)
        self._difficulty = float(value)
        _capi.check(self._lib.taco_env_set_difficulty(self._h, self._difficulty), "taco_env_set_difficulty")

    # ------------------------------------------------------------------ API
    def _clamped(self, t, lim):
        return t if math.isinf(lim) else torch.clamp(t, -lim, lim)

    def reset(self):
        """vec_task_asymmetry.py:352-361: returns the current (initially zero) buffers; the actual
        re-initialisation happens lazily at the start of the next step (reset_buf starts all ones)."""
        # Fresh tensors, like the reference's out-of-place clamp: PPO.run keeps these two as ITS persistent observation storage
        # (``obs.copy_(next_obs)``, ppo_asymmetry.py:297-299,328-329) and stores them AFTER env.step (:326); a view of the
        # library's history buffers would be overwritten by later steps.
        self.obs_dict["obs"] = torch.clamp(self.obs_buf, -self.clip_obs, self.clip_obs).to(self.rl_device)
        self.obs_dict["states"] = torch.clamp(self.states_buf, -self.clip_states, self.clip_states).to(self.rl_device)
        return self.obs_dict

    def step(self, actions):
        """vec_task_asymmetry.py:290-334.  ``actions``: (num_envs, 4) float32 CUDA tensor."""
        if not isinstance(actions, torch.Tensor):
            raise TypeError("actions must be a torch.Tensor")
        if actions.shape != (self.num_envs, self.num_acts):
            raise ValueError(f"actions must have shape {(self.num_envs, self.num_acts)}, got {tuple(actions.shape)}")
        if actions.device.type != "cuda" or (actions.device.index or 0) != self.device_id:
            actions = actions.to(self.device)
        if actions.dtype != torch.float32:
            actions = actions.float()
        if not actions.is_contiguous():          # gymtorch.unwrap_tensor raises here (gymtorch.py:98-99); we copy instead
            actions = actions.contiguous()
        self._actions_keepalive = actions
        stream = torch.cuda.current_stream(self.device_id).cuda_stream
        _capi.check(self._lib.taco_env_step(self._h, C.c_void_p(actions.data_ptr()), C.c_void_p(stream)), "taco_env_step")
        self._advance()
        self.extras["time_outs"] = self.timeout_buf.to(self.rl_device)
        self.obs_dict["obs"] = self._clamped(self.obs_buf, self.clip_obs).to(self.rl_device)
        self.obs_dict["states"] = self._clamped(self.states_buf, self.clip_states).to(self.rl_device)
        return self.obs_dict, self.rew_buf.to(self.rl_device), self.reset_buf.to(self.rl_device), self.extras

    def step_host(self, actions_host, rew_host=None, reset_host=None, time_outs_host=None):
        """One step through HOST buffers (pinned torch CPU tensors): H2D actions, kernel, D2H
        rew/reset/time_outs, stream sync -- the end-to-end path bench.py times."""
        stream = torch.cuda.current_stream(self.device_id).cuda_stream
        ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)
        _capi.check(self._lib.taco_env_step_host(self._h, ptr(actions_host), ptr(rew_host), ptr(reset_host),
                                                 ptr(time_outs_host), C.c_void_p(stream)), "taco_env_step_host")
        self._advance()

    def step_host_compact(self, actions_host, rew_host, flags_host):
        """``step_host`` with the compact result format: ``rew_host`` float32 (or None) and ``flags_host`` uint8 with bit 0 = reset,
        bit 1 = time-out (5 bytes device->host per env instead of 13).  Pinned host tensors only."""
        stream = torch.cuda.current_stream(self.device_id).cuda_stream
        ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)
        _capi.check(self._lib.taco_env_step_host_compact(self._h, ptr(actions_host), ptr(rew_host), ptr(flags_host), C.c_void_p(stream)),
                    "taco_env_step_host_compact")
        self._advance()

    def _advance(self):
        if self.rollout_buffer is not None:
            self._ring_cur += 1
        else:
            self._cur ^= 1
        self.step_count += 1

    # ------------------------------------------------------------------ zero-copy rollout storage
    def attach_rollout(self, buffer):
        """Let the step kernel write observation / state history, reward, done and time-out of every step straight into
        ``buffer`` (a taco_b200.RolloutBuffer): what PPOReplayBuffer.store copies per step (buffer_asymmetry.py:49-68)."""
        if (buffer.num_envs, buffer.obs_len, buffer.states_len, buffer.obs_dim, buffer.states_dim) != \
                (self.num_envs, self.len_obs, self.len_states, self.num_obs, self.num_states):
            raise ValueError("RolloutBuffer shape does not match the env")
        if buffer.device_id != self.device_id:
            raise ValueError("RolloutBuffer is on another device")
        if not (math.isinf(self.clip_obs) and math.isinf(self.clip_states)):
            # step() returns clamp(obs_buf) / clamp(states_buf) (vec_task_asymmetry.py:331-332); the ring holds the raw history that
            # actor, critic and the update read in place, so a finite clip would silently diverge from the drop-in path
            raise ValueError("attach_rollout: clipObservations / clipStates must be inf for the zero-copy rollout path")
        if self.rollout_buffer is not None:
            self.detach_rollout()
        stream = torch.cuda.current_stream(self.device_id).cuda_stream
        p = lambda t: C.c_void_p(t.data_ptr())
        _capi.check(self._lib.taco_env_attach_rollout(self._h, p(buffer.obs_ring), p(buffer.states_ring), buffer.horizon_len + 1,
                                                      p(buffer.rew_buf), p(buffer.done_buf), p(buffer.timeout_buf), C.c_void_p(stream)),
                    "taco_env_attach_rollout")
        self.rollout_buffer = buffer
        self._ring_cur = 0

    def rewind_rollout(self):
        """Start the next rollout: the newest slot becomes slot 0."""
        stream = torch.cuda.current_stream(self.device_id).cuda_stream
        _capi.check(self._lib.taco_env_rewind_rollout(self._h, C.c_void_p(stream)), "taco_env_rewind_rollout")
        self._ring_cur = 0

    # ------------------------------------------------------------------ CUDA-graph support
    def graph_begin(self):
        """Switch the step index to a device-side counter (taco_env_graph_begin) so that launches captured in a CUDA graph stay valid
        on replay; see ``taco_b200.rollout.GraphedRollout``."""
        stream = torch.cuda.current_stream(self.device_id).cuda_stream
        _capi.check(self._lib.taco_env_graph_begin(self._h, C.c_void_p(stream)), "taco_env_graph_begin")

    def graph_advance(self, steps):
        stream = torch.cuda.current_stream(self.device_id).cuda_stream
        _capi.check(self._lib.taco_env_graph_advance(self._h, int(steps), C.c_void_p(stream)), "taco_env_graph_advance")

    def graph_end(self):
        """Back to host-side counting; the step index is read back from the device (synchronises)."""
        stream = torch.cuda.current_stream(self.device_id).cuda_stream
        _capi.check(self._lib.taco_env_graph_end(self._h, C.c_void_p(stream)), "taco_env_graph_end")
        self.step_count = self.step_counter()[1]

    def step_counter(self):
        """(device address of the graph-mode step counter or 0, the library's host view of the step index)."""
        ptr, host = C.c_void_p(), C.c_uint32()
        _capi.check(self._lib.taco_env_step_counter(self._h, C.byref(ptr), C.byref(host)), "taco_env_step_counter")
        return (ptr.value or 0), int(host.value)

    def step_raw(self, actions):
        """``step`` without the return-value bookkeeping: one C call (contiguous float32 (num_envs, 4) CUDA tensor)."""
        stream = torch.cuda.current_stream(self.device_id).cuda_stream
        _capi.check(self._lib.taco_env_step(self._h, C.c_void_p(actions.data_ptr()), C.c_void_p(stream)), "taco_env_step")
        self._advance()

    def detach_rollout(self):
        stream = torch.cuda.current_stream(self.device_id).cuda_stream
        _capi.check(self._lib.taco_env_detach_rollout(self._h, C.c_void_p(stream)), "taco_env_detach_rollout")
        self.rollout_buffer = None
        self._ring_cur = 0

    def reset_all(self):
        stream = torch.cuda.current_stream(self.device_id).cuda_stream
        _capi.check(self._lib.taco_env_reset_all(self._h, C.c_void_p(stream)), "taco_env_reset_all")
        self._wrap_buffers()
        self._ring_cur = 0
        self.step_count = 0

    def set_seed(self, seed):
        self.seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        _capi.check(self._lib.taco_env_set_seed(self._h, self.seed), "taco_env_set_seed")

    def stats(self, out=None):
        """Rollout statistics since the last call as a float64 CUDA tensor of 8:
        [sum_reward, n_done, n_timeout, sum_ep_return, sum_ep_len, n_nonfinite, n_delay_overflow, n_env_steps]."""
        if out is None:
            out = torch.empty(_capi.NUM_STATS, dtype=torch.float64, device=self.device)
        stream = torch.cuda.current_stream(self.device_id).cuda_stream
        _capi.check(self._lib.taco_env_stats(self._h, C.c_void_p(out.data_ptr()), C.c_void_p(0), C.c_void_p(stream)), "taco_env_stats")
        return out

    def random_actions(self, step_index, out=None):
        """U(-1,1) actions from the Philox action stream (same draws as oracle.philox STREAM_ACTIONS)."""
        if out is None:
            out = torch.empty(self.num_envs, self.num_acts, dtype=torch.float32, device=self.device)
        stream = torch.cuda.current_stream(self.device_id).cuda_stream
        _capi.check(self._lib.taco_env_fill_random_actions(self._h, C.c_void_p(out.data_ptr()), int(step_index) & 0xFFFFFFFF,
                                                           C.c_void_p(stream)), "taco_env_fill_random_actions")
        return out

    def export_state(self):
        out = np.empty((self.num_envs, _capi.STATE_WORDS), dtype=np.float32)
        _capi.check(self._lib.taco_env_export_state(self._h, out.ctypes.data_as(C.c_void_p)), "taco_env_export_state")
        return out

    def record_state(self, ids, out=None):
        """Trajectory recorder (``taco_env_record_state``): the ``export_state`` rows of the local env ids ``ids`` (int32 CUDA tensor,
        (k,)) into ``out`` ((k, 64) float32 CUDA tensor) on the device, without a host sync (capturable in a CUDA graph)."""
        if ids.dtype != torch.int32 or ids.device.type != "cuda" or not ids.is_contiguous():
            raise ValueError("record_state: ids must be a contiguous int32 CUDA tensor")
        k = ids.numel()
        if out is None:
            out = torch.empty(k, _capi.STATE_WORDS, dtype=torch.float32, device=self.device)
        if out.dtype != torch.float32 or not out.is_contiguous() or out.numel() != k * _capi.STATE_WORDS:
            raise ValueError("record_state: out must be a contiguous float32 (k, 64) tensor")
        stream = torch.cuda.current_stream(self.device_id).cuda_stream
        _capi.check(self._lib.taco_env_record_state(self._h, C.c_void_p(ids.data_ptr()), k, C.c_void_p(out.data_ptr()), C.c_void_p(stream)),
                    "taco_env_record_state")
        return out

    def import_state(self, arr):
        arr = np.ascontiguousarray(arr, dtype=np.float32)
        assert arr.shape == (self.num_envs, _capi.STATE_WORDS)
        _capi.check(self._lib.taco_env_import_state(self._h, arr.ctypes.data_as(C.c_void_p)), "taco_env_import_state")

    def state_checkpoint(self):
        """The complete env state (everything the next ``step`` depends on) as one uint8 numpy array; see ``load_state_checkpoint``."""
        nbytes = C.c_uint64()
        _capi.check(self._lib.taco_env_checkpoint_size(self._h, C.byref(nbytes)), "taco_env_checkpoint_size")
        blob = np.empty(nbytes.value, dtype=np.uint8)
        _capi.check(self._lib.taco_env_checkpoint_save(self._h, blob.ctypes.data_as(C.c_void_p), nbytes.value), "taco_env_checkpoint_save")
        return blob

    def load_state_checkpoint(self, blob):
        """Restore a ``state_checkpoint()`` of an env with the same cfg: stepping continues bit-identically (same Philox step index,
        pending-action ring, history buffers, difficulty and seed)."""
        blob = np.ascontiguousarray(blob, dtype=np.uint8)
        _capi.check(self._lib.taco_env_checkpoint_load(self._h, blob.ctypes.data_as(C.c_void_p), blob.size), "taco_env_checkpoint_load")
        self._wrap_buffers()
        self.step_count = self.step_counter()[1]
        self._difficulty = self._read_difficulty()

    def _read_difficulty(self):
        d = C.c_float()
        _capi.check(self._lib.taco_env_get_difficulty(self._h, C.byref(d)), "taco_env_get_difficulty")
        return d.value

    def save_state(self, path):
        np.save(path, self.state_checkpoint(), allow_pickle=False)

    def load_state(self, path):
        self.load_state_checkpoint(np.load(path, allow_pickle=False))

    def debug_delay(self):
        out = np.empty((self.num_envs, self.control_freq_inv, 4), dtype=np.float32)
        _capi.check(self._lib.taco_env_debug_delay(self._h, out.ctypes.data_as(C.c_void_p)), "taco_env_debug_delay")
        return out

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.taco_env_destroy(self._h)
            self._h = C.c_void_p(0)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class FpvPos(FpvVecTask):
    task_mode = "pos"


class FpvRotate(FpvVecTask):
    task_mode = "rotate"


class FpvFlip(FpvVecTask):
    task_mode = "flip"


class FpvMix(FpvVecTask):
    task_mode = "mix"


# tasks/__init__.py:33-39
isaacgym_task_map = {"Fpv_pos": FpvPos, "Fpv_rotate": FpvRotate, "Fpv_flip": FpvFlip, "Fpv_mix": FpvMix}

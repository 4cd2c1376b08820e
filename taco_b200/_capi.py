"""ctypes binding of the C ABI in include/taco_b200.h (libtaco_b200.so).

This is the whole Python<->native boundary: plain pointers and sizes, no torch types.  It
plays the role gymtorch.wrap_tensor / unwrap_tensor play in the reference
(python/isaacgym/gymtorch.py:61-106): raw device pointers in, zero-copy torch views out.
The library must exist -- there is no CPU fallback; a missing or unloadable .so raises.
"""
import ctypes as C
import os

import numpy as np

_LIB_PATH = os.environ.get("TACO_B200_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib", "libtaco_b200.so")

ABI_VERSION = 1
TASK = {"pos": 0, "rotate": 1, "flip": 2, "mix": 3}
NUM_OBS, NUM_ACTS, NUM_STATS, STATE_WORDS = 26, 4, 8, 64
EPISODE_SUMMARY_WORDS = 15        # TACO_EPISODE_SUMMARY_WORDS: 3 tasks x [episodes, time-outs, sum length, sum ret, sum ret^2]

FLAGS = {  # cfg key -> bit (include/taco_b200.h TACO_F_*)
    "random_copter_pos": 1 << 0, "random_copter_quat": 1 << 1, "random_copter_vel": 1 << 2,
    "random_target_pos": 1 << 3, "random_target_yaw": 1 << 4, "battery_consumption": 1 << 5,
    "random_voltage": 1 << 6, "rotor_noise": 1 << 7, "rotor_response": 1 << 8,
    "random_rotordynamic_coe": 1 << 9, "random_rotor_response": 1 << 10, "random_rotor_speed": 1 << 11,
    "random_aerodynamic_coe": 1 << 12, "ramdom_delay_time": 1 << 13, "ramdom_deploy_time": 1 << 14,
    "random_command": 1 << 15, "observation_noise": 1 << 16,
}
F_STRICT_FP = 1 << 24
F_DEBUG_DELAY = 1 << 25


class TacoCfg(C.Structure):
    _fields_ = [
        ("abi_version", C.c_int32), ("num_envs", C.c_int32), ("env_offset", C.c_int64), ("num_envs_global", C.c_int64),
        ("task_mode", C.c_int32), ("len_obs", C.c_int32), ("len_states", C.c_int32), ("max_episode_length", C.c_int32),
        ("control_freq_inv", C.c_int32), ("substeps", C.c_int32), ("delay_time", C.c_int32), ("flags", C.c_uint32),
        ("dt", C.c_float), ("rotor_response_time", C.c_float), ("difficulty", C.c_float), ("clip_actions", C.c_float),
        ("seed", C.c_uint64),
    ]


class TacoBuffers(C.Structure):
    _fields_ = [
        ("obs", C.c_void_p), ("states", C.c_void_p), ("rew", C.c_void_p), ("reset", C.c_void_p),
        ("time_outs", C.c_void_p), ("progress", C.c_void_p), ("obs_ab", C.c_void_p * 2), ("states_ab", C.c_void_p * 2),
        ("num_envs", C.c_int32), ("len_obs", C.c_int32), ("len_states", C.c_int32), ("num_obs", C.c_int32),
    ]


_lib = None


def lib():
    """Load libtaco_b200.so (built by taco_b200.build / __graft_entry__.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise RuntimeError(f"{_LIB_PATH} is missing: run `python -m taco_b200.build` (there is no CPU fallback)")
    L = C.CDLL(_LIB_PATH)
    vp, i32, u32, u64, f32 = C.c_void_p, C.c_int32, C.c_uint32, C.c_uint64, C.c_float
    sig = {
        "taco_abi_version": (C.c_int, []),
        "taco_launch_count": (C.c_int, [C.POINTER(u64)]),
        "taco_last_error": (C.c_char_p, []),
        "taco_env_create": (C.c_int, [C.POINTER(TacoCfg), C.c_int, C.POINTER(vp)]),
        "taco_env_destroy": (C.c_int, [vp]),
        "taco_env_buffers": (C.c_int, [vp, C.POINTER(TacoBuffers)]),
        "taco_env_step": (C.c_int, [vp, vp, vp]),
        "taco_env_step_host": (C.c_int, [vp, vp, vp, vp, vp, vp]),
        "taco_env_step_host_compact": (C.c_int, [vp, vp, vp, vp, vp]),
        "taco_env_reset_all": (C.c_int, [vp, vp]),
        "taco_env_graph_begin": (C.c_int, [vp, vp]),
        "taco_env_graph_advance": (C.c_int, [vp, u32, vp]),
        "taco_env_graph_end": (C.c_int, [vp, vp]),
        "taco_env_step_counter": (C.c_int, [vp, C.POINTER(vp), C.POINTER(u32)]),
        "taco_actor_act_counter": (C.c_int, [vp, vp, i32, vp, C.c_int64, u64, u32, vp, vp, vp, vp, vp, i32, vp]),
        "taco_env_attach_rollout": (C.c_int, [vp, vp, vp, i32, vp, vp, vp, vp]),
        "taco_env_rewind_rollout": (C.c_int, [vp, vp]),
        "taco_env_detach_rollout": (C.c_int, [vp, vp]),
        "taco_env_rollout_cursor": (C.c_int, [vp]),
        "taco_env_states_strip": (C.c_int, [vp, C.POINTER(vp), C.POINTER(i32), C.POINTER(i32)]),
        "taco_env_set_difficulty": (C.c_int, [vp, f32]),
        "taco_env_set_seed": (C.c_int, [vp, u64]),
        "taco_env_stats": (C.c_int, [vp, vp, vp, vp]),
        "taco_env_fill_random_actions": (C.c_int, [vp, vp, u32, vp]),
        "taco_env_export_state": (C.c_int, [vp, vp]),
        "taco_env_import_state": (C.c_int, [vp, vp]),
        "taco_env_debug_delay": (C.c_int, [vp, vp]),
        "taco_env_attach_episode_log": (C.c_int, [vp, C.c_int64, vp]),
        "taco_env_detach_episode_log": (C.c_int, [vp]),
        "taco_env_episode_log_buffers": (C.c_int, [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(C.c_int64)]),
        "taco_env_episode_log_clear": (C.c_int, [vp, vp]),
        "taco_env_record_state": (C.c_int, [vp, vp, i32, vp, vp]),
        "taco_env_attach_rollout_episodes": (C.c_int, [vp, C.c_int64, vp]),
        "taco_env_detach_rollout_episodes": (C.c_int, [vp]),
        "taco_env_rollout_episodes_buffers": (C.c_int, [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(C.c_int64)]),
        "taco_env_rollout_episodes_clear": (C.c_int, [vp, vp]),
        "taco_env_scan_rollout_episodes": (C.c_int, [vp, vp, vp]),
        "taco_selftest_divc": (C.c_int, [C.c_int, f32, C.POINTER(u64)]),
        "taco_selftest_atan2": (C.c_int, [C.c_int, C.c_uint32, C.POINTER(f32), C.POINTER(C.c_uint32)]),
        "taco_actor_create": (C.c_int, [C.c_int, C.POINTER(i32), i32, C.POINTER(vp)]),
        "taco_actor_destroy": (C.c_int, [vp]),
        "taco_actor_load": (C.c_int, [vp, C.POINTER(vp), C.POINTER(vp), f32, vp]),
        "taco_actor_forward": (C.c_int, [vp, vp, vp, i32, i32, vp]),
        "taco_actor_sigmas": (C.c_int, [vp, vp]),
        "taco_actor_weights": (C.c_int, [vp, i32, vp, vp]),
        "taco_actor_tc_available": (C.c_int, [vp]),
        "taco_actor_set_log_std": (C.c_int, [vp, vp, vp]),
        "taco_env_get_difficulty": (C.c_int, [vp, C.POINTER(f32)]),
        "taco_env_checkpoint_size": (C.c_int, [vp, C.POINTER(u64)]),
        "taco_env_checkpoint_save": (C.c_int, [vp, vp, u64]),
        "taco_env_checkpoint_load": (C.c_int, [vp, vp, u64]),
        "taco_spectral_project": (C.c_int, [C.c_int, vp, i32, i32, f32, vp, vp]),
        "taco_actor_act": (C.c_int, [vp, vp, i32, vp, C.c_int64, u64, u32, vp, vp, vp, vp, i32, vp]),
        "taco_critic_create": (C.c_int, [C.c_int, i32, i32, i32, i32, C.POINTER(i32), i32, C.POINTER(vp)]),
        "taco_critic_destroy": (C.c_int, [vp]),
        "taco_critic_load": (C.c_int, [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), vp]),
        "taco_critic_tc_available": (C.c_int, [vp]),
        "taco_critic_forward": (C.c_int, [vp, vp, vp, i32, i32, vp]),
        "taco_ppo_create": (C.c_int, [C.c_int, vp, C.POINTER(vp)]),
        "taco_ppo_create_layers": (C.c_int, [C.c_int, vp, i32, C.POINTER(vp)]),
        "taco_ppo_destroy": (C.c_int, [vp]),
        "taco_ppo_num_params": (C.c_int, [vp, C.POINTER(C.c_int64)]),
        "taco_ppo_param_offsets": (C.c_int, [vp, C.POINTER(C.c_int64), i32, C.POINTER(i32)]),
        "taco_ppo_buffers": (C.c_int, [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(vp)]),
        "taco_ppo_params_changed": (C.c_int, [vp, vp]),
        "taco_ppo_begin_update": (C.c_int, [vp, vp]),
        "taco_ppo_forward_loss": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
        "taco_ppo_loss_sums": (C.c_int, [vp, C.POINTER(vp)]),
        "taco_ppo_decide": (C.c_int, [vp, vp, vp]),
        "taco_ppo_backward": (C.c_int, [vp, vp]),
        "taco_ppo_apply": (C.c_int, [vp, vp, vp]),
        "taco_ppo_end_update": (C.c_int, [vp, vp, i32, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), vp]),
        "taco_ppo_sigmas": (C.c_int, [vp, vp]),
        "taco_ppo_debug_outputs": (C.c_int, [vp, C.POINTER(vp), C.POINTER(vp)]),
        "taco_gemm_selftest": (C.c_int, [C.c_int, vp, vp, vp, i32, i32, i32, i32, vp]),
        "taco_gemm_selftest_mn": (C.c_int, [C.c_int, vp, vp, vp, i32, i32, i32, i32, vp]),
        "taco_gae_advantages": (C.c_int, [C.c_int, i32, i32, vp, vp, vp, vp, vp, f32, f32, vp, vp, vp, vp]),
        "taco_gae_normalize": (C.c_int, [C.c_int, vp, C.c_int64, vp, vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)          # AttributeError if the symbol is not exported
        fn.restype, fn.argtypes = res, args
    if L.taco_abi_version() != ABI_VERSION:
        raise RuntimeError("libtaco_b200.so ABI version mismatch; rebuild with `python -m taco_b200.build --force`")
    _lib = L
    return L


def check(rc, what):
    if rc != 0:
        msg = lib().taco_last_error()
        raise RuntimeError(f"{what} failed (code {rc}): {msg.decode() if msg else ''}")


class TacoPPOCfg(C.Structure):
    _fields_ = [("batch", C.c_int32), ("obs_dim", C.c_int32), ("act_dim", C.c_int32), ("state_dim", C.c_int32), ("seq_len", C.c_int32),
                ("lstm_hidden", C.c_int32), ("n_actor_hidden", C.c_int32), ("actor_hidden", C.c_int32 * 4),
                ("n_critic_hidden", C.c_int32), ("critic_hidden", C.c_int32 * 4)]


class TacoPPOHyper(C.Structure):
    _fields_ = [("lr", C.c_float), ("clip", C.c_float), ("target_kl", C.c_float), ("max_grad", C.c_float), ("pi_coef", C.c_float),
                ("vf_coef", C.c_float), ("ent_coef", C.c_float), ("lipschitz", C.c_float), ("use_lipschitz", C.c_int32), ("world", C.c_int32)]


# TacoEpisode (include/taco_b200.h), 48 bytes per record
EPISODE_DTYPE = np.dtype([("env_id", "<i8"), ("end_step", "<u4"), ("length", "<i4"), ("task", "<i2"), ("timed_out", "<i2"),
                          ("ret", "<f4"), ("pos_err_mean", "<f4"), ("pos_err_final", "<f4"), ("tilt_max", "<f4"),
                          ("speed_mean", "<f4"), ("angvel_max", "<f4"), ("roll_travel", "<f4")])
assert EPISODE_DTYPE.itemsize == 48

# TacoRolloutEpisode: the first six fields of TacoEpisode, 24 bytes per record
ROLLOUT_EPISODE_DTYPE = np.dtype(EPISODE_DTYPE.descr[:6])
assert ROLLOUT_EPISODE_DTYPE.itemsize == 24


class _CudaView:
    """Minimal __cuda_array_interface__ holder so torch can wrap a raw device pointer zero-copy
    (the ctypes analogue of gymtorch.wrap_tensor_impl, gymtorch.cpp:33-158)."""

    def __init__(self, ptr, shape, typestr, owner):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False), "version": 2}
        self._owner = owner          # keeps the env (and its arena) alive while the view exists


def wrap(ptr, shape, typestr, device, owner):
    import torch
    return torch.as_tensor(_CudaView(ptr, shape, typestr, owner), device=device)


def launch_count():
    """Kernel launches issued by libtaco_b200.so in this process so far."""
    n = C.c_uint64()
    check(lib().taco_launch_count(C.byref(n)), "taco_launch_count")
    return int(n.value)

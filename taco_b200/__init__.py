"""taco_b200 -- B200-native fused flight-dynamics / rollout step for the TACO fpv tasks.

Only what the hot path needs: csrc/ (sm_100a CUDA kernels + the C ABI), the ctypes binding,
and FpvVecTask, the host-side mirror of the reference VecTask interface.
"""
from .config import make_cfg, TASK_MODES  # noqa: F401
from .actor import ActorMLP, spectral_normalize_  # noqa: F401
from .critic import CriticLSTM  # noqa: F401
from .rollout import RolloutBuffer, RolloutEpisodes, collect_rollout, GraphedRollout  # noqa: F401
from . import ppo  # noqa: F401
from .evaluate import EpisodeLog, evaluate_policy, summarise_episodes, save_trajectories  # noqa: F401
from .fpv_vec_task import FpvVecTask, FpvPos, FpvRotate, FpvFlip, FpvMix, isaacgym_task_map, Box  # noqa: F401

__all__ = ["make_cfg", "TASK_MODES", "FpvVecTask", "FpvPos", "FpvRotate", "FpvFlip", "FpvMix", "isaacgym_task_map", "Box", "ActorMLP", "spectral_normalize_", "CriticLSTM", "RolloutBuffer", "RolloutEpisodes", "collect_rollout", "GraphedRollout",
           "EpisodeLog", "evaluate_policy", "summarise_episodes", "save_trajectories"]

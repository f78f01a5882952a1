"""multidronesim_b200 -- B200-native batched drone simulation hot path.

Host-side mirror of the reference's packages (envs, control, model, cbf, trajectories, obstacles,
utils) over a C-ABI library of hand-written sm_100a CUDA kernels (include/mds_b200.h)."""
from . import _lib
from .enums import DroneModel, Physics
from .constants import DroneConstants
from .envs import BatchedCtrlAviary, CtrlAviary
from .rollout import FusedRollout, HostPipeline, HostRollout, LearningRollout, PerCallPipeline, SwarmStreams, TorqueLearningRollout
from . import control, model, cbf, trajectories, obstacles, utils, dist, scenarios, fedce

__all__ = ["DroneModel", "Physics", "DroneConstants", "BatchedCtrlAviary", "CtrlAviary", "FusedRollout", "HostPipeline", "HostRollout", "LearningRollout", "PerCallPipeline", "SwarmStreams", "TorqueLearningRollout",
           "control", "model", "cbf", "trajectories", "obstacles", "utils", "dist", "scenarios", "_lib"]

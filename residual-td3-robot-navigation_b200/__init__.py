"""B200-native hot path of benmcclusky/Residual-TD3-Robot-Navigation.

`Environment` (environment.py of the reference) and, as they land, `ReplayBuffer` / `TD3` / `Robot`
(robot.py of the reference), all executing in csrc/librtd3.so - hand-written sm_100a CUDA behind a C ABI.
"""
from . import _lib, configuration, constants  # noqa: F401
from .environment import Environment, perlin_maps_device, synthetic_maps  # noqa: F401
from .rng import MtBank  # noqa: F401
from .learner import ReplayBuffer, Residual_Actor_Network, Residual_Critic_Network, TD3  # noqa: F401
from .robot import Robot  # noqa: F401
from .trainer import BatchedTrainer, DriverLoop, shard_range  # noqa: F401
from .checkpoint import PendingCheckpoint, load_checkpoint, save_checkpoint  # noqa: F401

__all__ = ["Environment", "MtBank", "synthetic_maps", "perlin_maps_device", "constants", "configuration", "ReplayBuffer",
           "Residual_Actor_Network", "Residual_Critic_Network", "TD3", "Robot", "BatchedTrainer", "DriverLoop", "shard_range",
           "save_checkpoint", "PendingCheckpoint", "load_checkpoint"]

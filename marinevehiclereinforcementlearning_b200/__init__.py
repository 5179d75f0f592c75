"""B200-native batched simulator for the BlueROV2 Heavy dynamics / Gym env
step of UnnamedMoose/MarineVehicleReinforcementLearning.

The compute path is hand-written sm_100a CUDA (``libmvrl.so``, C ABI in
``include/mvrl.h``); this package is the Python host side that mirrors the
reference's module / class / function names.  There is no CPU fallback.
"""
from . import _lib  # noqa: F401
from .auv import AuvCylVecEnv, AuvVecEnv, FlowField  # noqa: F401
from .policy import Actor, Critic, CriticTarget, MlpGaussianPolicy, SquashedGaussianPolicy, quantile_huber_loss  # noqa: F401
from .rov3 import BlueROV2Heavy3DoFVecEnv, Rov3Constants, Rov3Derivs  # noqa: F401
from .rov6 import BlueROV2Heavy6DoFVecEnv, Rov6Constants, Rov6Derivs  # noqa: F401
from .vec_tools import ReplayBuffer  # noqa: F401

__all__ = ["BlueROV2Heavy6DoFVecEnv", "Rov6Constants", "Rov6Derivs", "BlueROV2Heavy3DoFVecEnv", "Rov3Constants", "Rov3Derivs",
           "AuvVecEnv", "AuvCylVecEnv", "FlowField", "MlpGaussianPolicy", "SquashedGaussianPolicy", "Actor", "Critic", "CriticTarget",
           "quantile_huber_loss", "ReplayBuffer"]

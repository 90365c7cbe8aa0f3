"""B200-native batched QuadX hover / yaw simulator + PPO rollout engine.

Drop-in for the ``simulation/`` env path of Grzetan/FPV-drone-RL-agent: the
``QuadXHoverEnv`` gymnasium API of hover.py and the vectorised env that
train_hover.py builds, on hand-written sm_100a CUDA kernels behind the C-ABI of
``include/quadx_b200.h``.  No CPU fallback: the classes raise if
``libquadx_b200.so`` is not built or no CUDA device is present."""
from ._lib import QX_FRAME_MASK, QX_FRAME_RGBA, QX_OBS_BF16, QX_OBS_F32, QX_TASK_HOVER, QX_TASK_YAW, QxConfig, QxError, default_config  # noqa: F401
from .hover_env import STATE_FIELDS, Box, QuadXHoverEnv, QuadXHoverVecEnv, QuadXSim  # noqa: F401
from .yaw_env import DroneEnv, QuadXYawVecEnv  # noqa: F401

__all__ = [
    "QxConfig", "QxError", "default_config", "QuadXSim", "QuadXHoverVecEnv", "QuadXHoverEnv", "QuadXYawVecEnv", "DroneEnv", "Box", "STATE_FIELDS",
    "QX_TASK_HOVER", "QX_TASK_YAW", "QX_OBS_F32", "QX_OBS_BF16", "QX_FRAME_RGBA", "QX_FRAME_MASK",
]

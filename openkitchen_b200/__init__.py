"""openkitchen_b200 -- B200-native batched step loop for OpenKitchen's racing environment.

Only what the hot path needs: ``csrc/`` (sm_100a kernels + the C ABI of include/openkitchen_b200.h),
this ctypes front-end, the drop-in C++ shim (``shim/``) and the pybind module (``pybind/``).
"""
from ._capi import (  # noqa: F401
    BEV_LANE,
    BEV_OFF,
    BEV_WALL,
    BUF,
    BUFFERS,
    LIB_PATH,
    MOVE_ACCELERATION,
    MOVE_VELOCITY,
    RAYCAST_BEAM,
    RAYCAST_BRUTE,
    RAYCAST_GRID,
    REWARD_CMAES_PROGRESS,
    REWARD_CONSTANT,
    REWARD_DISPLACEMENT,
    REWARD_LANE_CENTER,
    REWARD_MIN_RAY,
    REWARD_NONE,
    REWARD_Q_PROGRESS,
    REWARD_TRACK_INDEX,
    RESET_DRAW_HEADING,
    RESET_DRAW_LANE,
    RESET_DRAW_POINT,
    OkError,
)
from . import dlpack  # noqa: F401
from .env import (  # noqa: F401
    Env,
    dequantize_obs_q16,
    pcie_probe,
    pinned_array,
    quantize_obs_q16,
    ray_fan,
    release_caches,
    track_columns,
    track_names,
    write_track_csv,
)

__version__ = "0.1.0"


def __getattr__(name):  # BatchEnv needs torch; keep the ctypes layer importable without it
    if name == "BatchEnv":
        from .batch_env import BatchEnv

        return BatchEnv
    raise AttributeError(name)

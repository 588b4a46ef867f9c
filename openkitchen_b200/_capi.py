"""ctypes bindings of include/openkitchen_b200.h (the product C ABI).

Loads ``openkitchen_b200/lib/libopenkitchen_b200.so`` (built in-tree by ``__graft_entry__.build()``
or ``make -C openkitchen_b200/csrc``).  There is no fallback: a missing library raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("OK_B200_LIB") or os.path.join(_HERE, "lib", "libopenkitchen_b200.so")

OK_SUCCESS = 0
OK_ERR_INVALID_ARG, OK_ERR_CUDA, OK_ERR_IO, OK_ERR_STATE, OK_ERR_CAPACITY, OK_ERR_NO_DEVICE = -1, -2, -3, -4, -5, -6

MOVE_VELOCITY, MOVE_ACCELERATION = 0, 1
REWARD_NONE, REWARD_Q_PROGRESS, REWARD_CMAES_PROGRESS, REWARD_CONSTANT = 0, 1, 2, 3
REWARD_DISPLACEMENT, REWARD_MIN_RAY, REWARD_TRACK_INDEX, REWARD_LANE_CENTER = 4, 5, 6, 7
RAYCAST_GRID, RAYCAST_BRUTE, RAYCAST_BEAM = 0, 1, 2
BEV_OFF, BEV_WALL, BEV_LANE = 0, 1, 2
RESET_DRAW_POINT, RESET_DRAW_LANE, RESET_DRAW_HEADING = 1, 2, 4

BUFFERS = [
    "pos_x", "pos_y", "rot", "speed", "accel", "act_throttle", "act_steer",
    "crashed", "timed_out", "done", "ss_ctr", "ss_x", "ss_y", "track_id",
    "hit_abs", "hit_rel", "obs", "hit_seg", "hit_t", "min_dist2",
    "nearest_idx", "prev_idx", "reward", "fitness", "reset_pt", "start_x", "start_y",
]
BUF = {n: i for i, n in enumerate(BUFFERS)}
DTYPE_F32, DTYPE_I32, DTYPE_U32, DTYPE_U8 = 0, 1, 2, 3

TRACK_ARRAYS = {
    "x": 0, "y": 1, "w_right": 2, "w_left": 3, "heading": 4,
    "li": 5, "lo": 6, "ri": 7, "ro": 8, "segments": 9,
}


class OkConfig(C.Structure):
    _fields_ = [
        ("device", C.c_int32),
        ("movement_mode", C.c_int32),
        ("reward_mode", C.c_int32),
        ("raycast_mode", C.c_int32),
        ("auto_reset", C.c_int32),
        ("auto_reset_stride", C.c_int32),
        ("sensor_range", C.c_float),
        ("speed_limit", C.c_float),
        ("dt", C.c_float),
        ("collision_dist2", C.c_float),
        ("sensor_offset", C.c_float),
        ("standstill_period", C.c_uint32),
        ("standstill_threshold", C.c_float),
        ("grid_cell", C.c_float),
        ("beam_cell", C.c_float),
        ("beam_bins", C.c_int32),
        ("agent_id_base", C.c_uint64),
    ]


class OkResetDraws(C.Structure):
    _fields_ = [("seed", C.c_uint32), ("flags", C.c_int32)]


class OkLaps(C.Structure):
    _fields_ = [("enabled", C.c_int32), ("target", C.c_int32)]


class OkLapBuffers(C.Structure):
    _fields_ = [("lap_idx", C.c_void_p), ("progress", C.c_void_p), ("laps", C.c_void_p), ("ticks", C.c_void_p),
                ("lap_start", C.c_void_p), ("last_lap", C.c_void_p), ("completed", C.c_void_p)]


class OkRaces(C.Structure):
    _fields_ = [("group", C.c_int32), ("flags", C.c_int32), ("radius", C.c_float)]


class OkRaceBuffers(C.Structure):
    _fields_ = [("hit_car", C.c_void_p), ("contact", C.c_void_p)]


RACE_SENSE, RACE_CONTACT = 1, 2  # OK_RACE_SENSE, OK_RACE_CONTACT


# the lap arrays of OkLapBuffers: field -> numpy dtype
LAP_ARRAYS = {"lap_idx": "int32", "progress": "int32", "laps": "int32", "ticks": "uint32", "lap_start": "uint32",
              "last_lap": "uint32", "completed": "uint8"}


class OkTrackInfo(C.Structure):
    _fields_ = [
        ("n_points", C.c_int32),
        ("n_segments", C.c_int32),
        ("grid_nx", C.c_int32),
        ("grid_ny", C.c_int32),
        ("grid_items", C.c_int32),
        ("blob_bytes", C.c_int32),
        ("grid_x0", C.c_float),
        ("grid_y0", C.c_float),
        ("grid_cell", C.c_float),
    ]


class OkPopulationCounters(C.Structure):
    _fields_ = [("agents", C.c_uint64), ("alive", C.c_uint64), ("crashed", C.c_uint64), ("timed_out", C.c_uint64), ("done", C.c_uint64)]


class OkLaunchStats(C.Structure):
    _fields_ = [
        ("kernel_launches", C.c_uint64),
        ("grid_blocks", C.c_int32),
        ("block_threads", C.c_int32),
        ("smem_bytes", C.c_int32),
        ("tiles", C.c_int32),
    ]


class OkPackedLayout(C.Structure):
    _fields_ = [("state_bytes", C.c_size_t), ("state_offset", C.c_size_t * 13), ("hits_bytes", C.c_size_t),
                ("hit_abs_offset", C.c_size_t), ("hit_rel_offset", C.c_size_t)]


class OkActorIO(C.Structure):
    _fields_ = [
        ("d_w1", C.c_void_p), ("d_b1", C.c_void_p), ("d_w2", C.c_void_p), ("d_b2", C.c_void_p),
        ("hidden", C.c_int32), ("n_actions", C.c_int32),
        ("d_action_table", C.c_void_p), ("d_uniform", C.c_void_p),
        ("greedy", C.c_int32), ("reserved", C.c_int32),
        ("d_action", C.c_void_p), ("d_log_prob", C.c_void_p), ("d_probs", C.c_void_p), ("d_obs", C.c_void_p),
        ("d_prev_reward", C.c_void_p), ("d_prev_done", C.c_void_p),
    ]


class OkLidarQuery(C.Structure):
    _fields_ = [
        ("x", C.c_void_p), ("y", C.c_void_p), ("rot", C.c_void_p), ("track_id", C.c_void_p),
        ("n", C.c_int64),
        ("ray_deg", C.c_void_p),
        ("rays", C.c_int32), ("reserved", C.c_int32),
        ("hit_abs", C.c_void_p), ("hit_rel", C.c_void_p), ("obs", C.c_void_p), ("hit_t", C.c_void_p),
        ("hit_seg", C.c_void_p), ("min_dist2", C.c_void_p), ("crashed", C.c_void_p),
    ]


class OkBevQuery(C.Structure):
    _fields_ = [
        ("x", C.c_void_p), ("y", C.c_void_p), ("rot", C.c_void_p), ("track_id", C.c_void_p),
        ("n", C.c_int64),
        ("height", C.c_int32), ("width", C.c_int32),
        ("scale", C.c_float), ("ahead", C.c_float),
        ("out", C.c_void_p),
    ]


# every symbol include/openkitchen_b200.h declares: (restype, argtypes)
_P = C.c_void_p
SIGNATURES = {
    "ok_abi_version": (C.c_int, []),
    "ok_last_error": (C.c_char_p, []),
    "ok_config_default": (None, [C.POINTER(OkConfig)]),
    "ok_create": (C.c_int, [C.POINTER(OkConfig), C.POINTER(_P)]),
    "ok_destroy": (None, [_P]),
    "ok_update_config": (C.c_int, [_P, C.POINTER(OkConfig)]),
    "ok_get_config": (C.c_int, [_P, C.POINTER(OkConfig)]),
    "ok_add_track": (C.c_int, [_P, _P, _P, _P, _P, C.c_int32, C.POINTER(C.c_int32)]),
    "ok_load_track_csv": (C.c_int, [_P, C.c_char_p, C.POINTER(C.c_int32)]),
    "ok_num_tracks": (C.c_int, [_P]),
    "ok_track_info": (C.c_int, [_P, C.c_int32, C.POINTER(OkTrackInfo)]),
    "ok_track_copy": (C.c_int64, [_P, C.c_int32, C.c_int32, _P, C.c_int64]),
    "ok_alloc_agents": (C.c_int, [_P, C.c_int64, C.c_int32, _P, _P]),
    "ok_num_agents": (C.c_int64, [_P]),
    "ok_num_rays": (C.c_int32, [_P]),
    "ok_reset_agents": (C.c_int, [_P, _P, _P, _P, _P, C.c_int64, _P]),
    "ok_reset_agents_host": (C.c_int, [_P, _P, _P, _P, _P, C.c_int64, _P]),
    "ok_set_reset_draws": (C.c_int, [_P, C.POINTER(OkResetDraws)]),
    "ok_get_reset_draws": (C.c_int, [_P, C.POINTER(OkResetDraws)]),
    "ok_reset_agents_drawn": (C.c_int, [_P, _P, _P, C.c_int64, _P]),
    "ok_reset_agents_drawn_host": (C.c_int, [_P, _P, _P, C.c_int64, _P]),
    "ok_reset_draw_counts": (C.c_int, [_P, C.POINTER(_P)]),
    "ok_set_laps": (C.c_int, [_P, C.POINTER(OkLaps), _P]),
    "ok_get_laps": (C.c_int, [_P, C.POINTER(OkLaps)]),
    "ok_lap_buffers": (C.c_int, [_P, C.POINTER(OkLapBuffers)]),
    "ok_set_races": (C.c_int, [_P, C.POINTER(OkRaces)]),
    "ok_get_races": (C.c_int, [_P, C.POINTER(OkRaces)]),
    "ok_race_buffers": (C.c_int, [_P, C.POINTER(OkRaceBuffers)]),
    "ok_cast_rays": (C.c_int, [_P, _P]),
    "ok_launch_step": (C.c_int, [_P, _P, _P, _P]),
    "ok_launch_steps_random": (C.c_int, [_P, C.c_uint64, C.c_int32, C.c_uint32, _P]),
    "ok_fill_random_actions": (C.c_int, [_P, C.c_uint64, C.c_uint32, _P]),
    "ok_genetic_policy": (C.c_int, [_P, _P, _P, C.c_int32, _P]),
    "ok_step_host": (C.c_int, [_P, _P, _P, _P, _P, _P, _P]),
    "ok_step_host_q16": (C.c_int, [_P, _P, _P, _P, _P, _P, _P]),
    "ok_packed_layout": (C.c_int, [_P, C.POINTER(OkPackedLayout)]),
    "ok_step_packed": (C.c_int, [_P, _P, _P, C.c_int32, _P]),
    "ok_host_alloc": (C.c_int, [C.POINTER(_P), C.c_size_t]),
    "ok_host_free": (C.c_int, [_P]),
    "ok_get_buffer": (C.c_int, [_P, C.c_int32, C.POINTER(_P), C.POINTER(C.c_int64), C.POINTER(C.c_int32)]),
    "ok_read_buffer": (C.c_int, [_P, C.c_int32, _P, C.c_size_t, _P]),
    "ok_write_buffer": (C.c_int, [_P, C.c_int32, _P, C.c_size_t, _P]),
    "ok_sync": (C.c_int, [_P, _P]),
    "ok_launch_stats": (C.c_int, [_P, C.POINTER(OkLaunchStats)]),
    "ok_population_counters": (C.c_int, [_P, C.POINTER(OkPopulationCounters), _P]),
    "ok_debug_stats": (C.c_int, [_P, C.POINTER(C.c_uint64), C.c_int32]),
    "ok_debug_violations": (C.c_int, [_P, C.POINTER(C.c_uint64), C.POINTER(C.c_int32)]),
    "ok_debug_trace": (C.c_int64, [_P, _P, C.c_int64, C.c_int32]),
    "ok_debug_tiles": (C.c_int64, [_P, _P, C.c_int64]),
    "ok_balance_schedule": (C.c_int, [_P, _P, _P]),
    "ok_eval_sincosf": (C.c_int, [_P, _P, _P, _P, C.c_int64]),
    "ok_beam_lookup": (C.c_int32, [_P, C.c_int32, C.c_float, C.c_float, C.c_float, _P, C.c_int32, C.POINTER(C.c_float)]),
    "ok_beam_lookup_ex": (C.c_int32, [_P, C.c_int32, C.c_float, C.c_float, C.c_float, _P, C.c_int32, C.POINTER(C.c_float),
                                      C.POINTER(C.c_float), C.POINTER(C.c_int32)]),
    "ok_beam_table_bytes": (C.c_int64, [_P, C.c_int32]),
    "ok_release_caches": (None, []),
    "ok_cmaes_controller": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_float, C.c_float, _P]),
    "ok_ppo_actor": (C.c_int, [_P, C.POINTER(OkActorIO), C.c_uint64, C.c_uint32, _P]),
    "ok_ppo_actor_step": (C.c_int, [_P, C.POINTER(OkActorIO), C.c_uint64, C.c_uint32, _P]),
    "ok_discounted_returns": (C.c_int, [_P, _P, _P, _P, C.c_int32, C.c_int64, C.c_float, _P]),
    "ok_track_query": (C.c_int, [_P, _P, _P, _P, C.c_int64, _P, _P, _P, _P]),
    "ok_track_query_host": (C.c_int, [_P, _P, _P, _P, C.c_int64, _P, _P, _P, _P]),
    "ok_lidar_query": (C.c_int, [_P, C.POINTER(OkLidarQuery), _P]),
    "ok_lidar_query_host": (C.c_int, [_P, C.POINTER(OkLidarQuery), _P]),
    "ok_bev_query": (C.c_int, [_P, C.POINTER(OkBevQuery), _P]),
    "ok_bev_query_host": (C.c_int, [_P, C.POINTER(OkBevQuery), _P]),
    "ok_pcie_probe": (C.c_int, [C.c_int32, C.c_size_t, C.c_int32, C.c_int32, C.POINTER(C.c_double)]),
}

_lib = None


class OkError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"openkitchen_b200 error {code}: {msg}")
        self.code = code


def load() -> C.CDLL:
    """Load the product library; raises if it has not been built (no fallback path exists)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "or `make -C openkitchen_b200/csrc`. openkitchen_b200 has no CPU fallback."
            )
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            try:
                fn = getattr(lib, name)
            except AttributeError:
                if os.environ.get("OK_B200_LIB"):  # an experiment build (older ABI) may lack the newest entry points
                    continue
                raise
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


def check(rc: int) -> int:
    if rc < 0:
        raise OkError(rc, (load().ok_last_error() or b"").decode())
    return rc

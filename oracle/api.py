"""ctypes front-end for the parity oracles (TEST INFRASTRUCTURE ONLY).

Two libraries export the same C API (oracle/ok_oracle.h):

* ``liboracle.so``       -- prefix ``oko_``: the plain-C restatement (oracle/ok_oracle.c)
* ``_ref/libokref.so``   -- prefix ``okr_``: the reference's own Agent.cpp / RaceTrack.cpp objects
                            driven by oracle/ref_harness.cpp

Only tests/, ``__graft_entry__.smoke()`` and bench.py's ``cpu_baseline`` / ``--impl reference``
legs may import this module; the product package never does.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))

BUF = {
    name: i
    for i, name in enumerate(
        [
            "pos_x", "pos_y", "rot", "speed", "accel", "act_throttle", "act_steer",
            "crashed", "timed_out", "done", "ss_ctr", "ss_x", "ss_y", "track_id",
            "hit_abs", "hit_rel", "obs", "hit_seg", "hit_t", "min_dist2",
            "nearest_idx", "prev_idx", "reward", "fitness", "reset_pt", "start_x", "start_y",
        ]
    )
}
U8_BUFS = {"crashed", "timed_out", "done"}
I32_BUFS = {"track_id", "hit_seg", "nearest_idx", "prev_idx", "reset_pt"}
U32_BUFS = {"ss_ctr"}
RAY_BUFS = {"obs": 1, "hit_seg": 1, "hit_t": 1, "hit_abs": 2, "hit_rel": 2}

TRACK_ARRAYS = {"x": 0, "y": 1, "w_right": 2, "w_left": 3, "heading": 4, "li": 5, "lo": 6, "ri": 7, "ro": 8, "segments": 9}


class OkoConfig(C.Structure):
    _fields_ = [
        ("movement_mode", C.c_int32),
        ("reward_mode", C.c_int32),
        ("auto_reset", C.c_int32),
        ("auto_reset_stride", C.c_int32),
        ("sensor_range", C.c_float),
        ("speed_limit", C.c_float),
        ("dt", C.c_float),
        ("collision_dist2", C.c_float),
        ("sensor_offset", C.c_float),
        ("standstill_period", C.c_uint32),
        ("standstill_threshold", C.c_float),
        ("pad_", C.c_uint32),
        ("agent_id_base", C.c_uint64),
    ]


def build(force: bool = False) -> None:
    """Compile the checkers (``make -C oracle``).  Building the checker is not using it."""
    ref = os.environ.get("OPENKITCHEN_REF")  # a checkout of the original project (see oracle/Makefile)
    if force or not os.path.exists(os.path.join(HERE, "liboracle.so")) or (
        ref and os.path.isdir(os.path.join(ref, "Environment")) and not os.path.exists(os.path.join(HERE, "_ref", "libokref.so"))
    ):
        subprocess.run(["make", "-C", HERE], check=True, capture_output=True)


def have_ref() -> bool:
    return os.path.exists(os.path.join(HERE, "_ref", "libokref.so"))


def _fp(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


class Oracle:
    """One oracle environment.  ``kind`` = ``"port"`` (C restatement) or ``"reference"`` (_ref objects)."""

    def __init__(self, kind: str = "port", **cfg):
        self.kind = kind
        if kind == "port":
            path, self.p = os.path.join(HERE, "liboracle.so"), "oko_"
        elif kind == "reference":
            path, self.p = os.path.join(HERE, "_ref", "libokref.so"), "okr_"
        else:
            raise ValueError(kind)
        if not os.path.exists(path):
            raise FileNotFoundError(f"{path} missing: run `make -C oracle`")
        self.lib = C.CDLL(path)
        f = self._f
        f("config_default", None, [C.POINTER(OkoConfig)])
        f("create", C.c_void_p, [C.POINTER(OkoConfig)])
        f("destroy", None, [C.c_void_p])
        f("update_config", None, [C.c_void_p, C.POINTER(OkoConfig)])
        f("set_threads", None, [C.c_int])
        f("get_max_threads", C.c_int, [])
        f("add_track", C.c_int, [C.c_void_p] * 5 + [C.c_int])
        f("load_track_csv", C.c_int, [C.c_void_p, C.c_char_p])
        f("num_tracks", C.c_int, [C.c_void_p])
        f("track_points", C.c_int, [C.c_void_p, C.c_int])
        f("track_segments", C.c_int, [C.c_void_p, C.c_int])
        f("track_array", C.c_void_p, [C.c_void_p, C.c_int, C.c_int])
        f("alloc_agents", C.c_int, [C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p])
        f("num_agents", C.c_int64, [C.c_void_p])
        f("buffer", C.c_void_p, [C.c_void_p, C.c_int])
        f("reset_agents", None, [C.c_void_p] * 5 + [C.c_int64])
        f("cast_rays", None, [C.c_void_p])
        f("step", None, [C.c_void_p] * 3)
        f("fill_random_actions", None, [C.c_void_p, C.c_uint64, C.c_uint32])
        f("sincosf", None, [C.c_float, C.POINTER(C.c_float), C.POINTER(C.c_float)])
        f("nearest_index", C.c_int32, [C.c_void_p, C.c_int, C.c_float, C.c_float])
        f("dist_lane_center", C.c_float, [C.c_void_p, C.c_int, C.c_float, C.c_float])
        f("dist_boundary", C.c_float, [C.c_void_p, C.c_int, C.c_float, C.c_float])
        f("normalize_angle_deg", C.c_float, [C.c_float])
        f("philox4x32_10", None, [C.c_void_p] * 3)
        c = OkoConfig()
        self._config_default(C.byref(c))
        for k, v in cfg.items():
            if not hasattr(c, k):
                raise AttributeError(k)
            setattr(c, k, v)
        self.cfg = c
        self.h = self._create(C.byref(c))
        self.n = 0
        self.rays = 0

    def _f(self, name, res, args):
        fn = getattr(self.lib, self.p + name)
        fn.restype, fn.argtypes = res, args
        setattr(self, "_" + name, fn)

    def close(self):
        if getattr(self, "h", None):
            self._destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def update_config(self, **cfg):
        """push self.cfg (after editing it, or with keyword overrides) into the live env"""
        for k, v in cfg.items():
            if not hasattr(self.cfg, k):
                raise AttributeError(k)
            setattr(self.cfg, k, v)
        self._update_config(self.h, C.byref(self.cfg))

    # ---- tracks -------------------------------------------------------------------------
    def add_track(self, cols) -> int:
        x, y, wr, wl = (np.ascontiguousarray(c, dtype=np.float32) for c in cols)
        tid = self._add_track(self.h, _fp(x), _fp(y), _fp(wr), _fp(wl), len(x))
        if tid < 0:
            raise RuntimeError("add_track failed")
        return tid

    def load_track_csv(self, path: str) -> int:
        tid = self._load_track_csv(self.h, path.encode())
        if tid < 0:
            raise RuntimeError(f"load_track_csv({path}) failed")
        return tid

    def track_points(self, t):
        return self._track_points(self.h, t)

    def track_segments(self, t):
        return self._track_segments(self.h, t)

    def track_array(self, t, name) -> np.ndarray:
        n, ns = self.track_points(t), self.track_segments(t)
        shape = {"li": (n, 2), "lo": (n, 2), "ri": (n, 2), "ro": (n, 2), "segments": (ns, 4)}.get(name, (n,))
        ptr = self._track_array(self.h, t, TRACK_ARRAYS[name])
        cnt = int(np.prod(shape))
        return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(C.c_float)), shape=(cnt,)).reshape(shape).copy()

    # ---- agents -------------------------------------------------------------------------
    def alloc_agents(self, n, ray_deg, track_id=None):
        ray_deg = np.ascontiguousarray(ray_deg, dtype=np.float32)
        tid = None if track_id is None else np.ascontiguousarray(track_id, dtype=np.int32)
        if self._alloc_agents(self.h, n, len(ray_deg), _fp(ray_deg), _fp(tid)) != 0:
            raise RuntimeError("alloc_agents failed")
        self.n, self.rays = n, len(ray_deg)

    def buffer(self, name) -> np.ndarray:
        """Zero-copy numpy view of a state / output buffer."""
        ptr = self._buffer(self.h, BUF[name])
        if name in U8_BUFS:
            ct, dt = C.c_uint8, np.uint8
        elif name in I32_BUFS:
            ct, dt = C.c_int32, np.int32
        elif name in U32_BUFS:
            ct, dt = C.c_uint32, np.uint32
        else:
            ct, dt = C.c_float, np.float32
        if name in RAY_BUFS:
            shape = (self.n, self.rays) if RAY_BUFS[name] == 1 else (self.n, self.rays, 2)
        else:
            shape = (self.n,)
        cnt = int(np.prod(shape))
        return np.ctypeslib.as_array(C.cast(ptr, C.POINTER(ct)), shape=(cnt,)).reshape(shape)

    def reset(self, agent_idx, pt_idx, lane_alpha=None, heading_off=None):
        ai = None if agent_idx is None else np.ascontiguousarray(agent_idx, dtype=np.int64)
        pt = np.ascontiguousarray(pt_idx, dtype=np.int32)
        la = None if lane_alpha is None else np.ascontiguousarray(lane_alpha, dtype=np.float32)
        ho = None if heading_off is None else np.ascontiguousarray(heading_off, dtype=np.float32)
        self._reset_agents(self.h, _fp(ai), _fp(pt), _fp(la), _fp(ho), len(pt))

    def cast_rays(self):
        self._cast_rays(self.h)

    def step(self, thr=None, steer=None):
        t = None if thr is None else np.ascontiguousarray(thr, dtype=np.float32)
        s = None if steer is None else np.ascontiguousarray(steer, dtype=np.float32)
        self._step(self.h, _fp(t), _fp(s))

    def fill_random_actions(self, step, seed=0x0C17C4E2):
        self._fill_random_actions(self.h, step, seed)

    def set_threads(self, n):
        self._set_threads(n)

    def max_threads(self):
        return self._get_max_threads()

    # ---- scalars ------------------------------------------------------------------------
    def sincosf(self, x):
        s, c = C.c_float(), C.c_float()
        self._sincosf(C.c_float(x), C.byref(s), C.byref(c))
        return s.value, c.value

    def nearest_index(self, t, x, y):
        return self._nearest_index(self.h, t, x, y)

    def dist_lane_center(self, t, x, y):
        return self._dist_lane_center(self.h, t, x, y)

    def dist_boundary(self, t, x, y):
        return self._dist_boundary(self.h, t, x, y)

    def normalize_angle_deg(self, a):
        return self._normalize_angle_deg(a)

    def philox(self, ctr, key):
        c = np.asarray(ctr, dtype=np.uint32)
        k = np.asarray(key, dtype=np.uint32)
        o = np.zeros(4, dtype=np.uint32)
        self._philox4x32_10(_fp(c), _fp(k), _fp(o))
        return o


def ray_fan(n_rays: int) -> np.ndarray:
    """deg_i = -70 + i*140/(R-1) in binary32, the generator of main_torch.cpp:26-34."""
    if n_rays == 1:
        return np.zeros(1, dtype=np.float32)
    i = np.arange(n_rays, dtype=np.int32).astype(np.float32)
    return (np.float32(-70.0) + (i * np.float32(140.0)) / np.float32(n_rays - 1)).astype(np.float32)


Q_LEARNING_FAN = np.array([-70.0, -30.0, 0.0, 30.0, 70.0], dtype=np.float32)  # QAgent.hpp:56-62
DEFAULT_FAN = np.arange(-70, 71, 10).astype(np.float32)  # Agent.cpp:13-17

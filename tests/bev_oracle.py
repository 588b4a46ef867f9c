"""The brute-force bird's-eye-view oracle (TEST INFRASTRUCTURE ONLY): tests/bev_oracle.c compiled into a temporary
directory on first use, driven with the port oracle's tracks and its sincosf restatement (oracle/api.py)."""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

from oracle.api import Oracle

HERE = os.path.dirname(os.path.abspath(__file__))
K_DEG2RAD = np.float32(np.pi / 180.0)  # float(M_PI / 180.0), as the oracle's K_DEG2RAD and the kernels' OK_DEG2RAD
_lib = None


def _load():
    """compile bev_oracle.c with the oracle's flags (oracle/Makefile: no contraction, -mfma for nothing but explicit fma)"""
    global _lib
    if _lib is None:
        cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else shutil.which("gcc")  # a distro gcc with libgomp
        out = os.path.join(tempfile.mkdtemp(prefix="ok_bev_oracle_"), "libbevoracle.so")
        subprocess.run([cc, "-O2", "-fPIC", "-mfma", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-Wall", "-shared",
                        "-o", out, os.path.join(HERE, "bev_oracle.c")], check=True, capture_output=True)
        lib = C.CDLL(out)
        lib.bev_oracle.restype = None
        lib.bev_oracle.argtypes = [C.c_void_p] * 4 + [C.c_int] + [C.c_float] * 4 + [C.c_int, C.c_int, C.c_float, C.c_float,
                                                                                  C.c_void_p]
        _lib = lib
    return _lib


class BevOracle(Oracle):
    """The port oracle with ``bev``: the brute-force raster ok_bev_query must reproduce bit for bit."""

    def __init__(self, **cfg):
        super().__init__("port", **cfg)
        self._loops = {}

    def bev(self, track, x, y, rot, height, width, scale, ahead=0.0) -> np.ndarray:
        """the raster at each pose (x, y, rot: scalars or 1-d arrays of one length) -> u8[n, height, width].  track: an id
        or one per pose, clamped to the tracks added as ok_bev_query clamps it."""
        lib = _load()
        x, y, rot = (np.atleast_1d(np.asarray(a, dtype=np.float32)) for a in (x, y, rot))
        nt = self._num_tracks(self.h)
        tid = np.clip(np.broadcast_to(np.asarray(track, dtype=np.int64), x.shape), 0, nt - 1)
        out = np.empty((len(x), height, width), dtype=np.uint8)
        for k in range(len(x)):
            t = int(tid[k])
            if t not in self._loops:
                self._loops[t] = [np.ascontiguousarray(self.track_array(t, nm), dtype=np.float32) for nm in ("li", "lo", "ri", "ro")]
            loops = self._loops[t]
            rs, rc = self.sincosf(K_DEG2RAD * rot[k])  # binary32 product, then the oracle's sincosf
            lib.bev_oracle(*(a.ctypes.data for a in loops), len(loops[0]), float(x[k]), float(y[k]), rs, rc, height, width,
                           float(np.float32(scale)), float(np.float32(ahead)), out[k].ctypes.data)
        return out

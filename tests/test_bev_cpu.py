"""CPU: the bird's-eye-view query's public surface and its oracle -- the ctypes OkBevQuery has the C layout, both entry
points refuse an env without a device, the Python wrappers reject malformed arguments before they reach the library, and
the brute-force oracle the GPU tests compare with (tests/bev_oracle.c) agrees with an independent float64 even-odd
classification everywhere but within 1e-3 px of a loop edge, and calls every centre-line point of the 23 tracks LANE."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

import openkitchen_b200 as ok
from openkitchen_b200 import _capi
from openkitchen_b200.batch_env import BatchEnv
from tests.bev_oracle import BevOracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = [f for f, _ in _capi.OkBevQuery._fields_]
LOOPS = ("li", "lo", "ri", "ro")


@pytest.mark.skipif(shutil.which("g++") is None, reason="needs g++")
def test_ctypes_layout_matches_the_header(tmp_path):
    src = tmp_path / "layout.c"
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "openkitchen_b200.h"', "int main(void) {",
             '  printf("%zu\\n", sizeof(OkBevQuery));']
    lines += [f'  printf("%zu\\n", offsetof(OkBevQuery, {f}));' for f in FIELDS]
    lines += ['  printf("%d %d %d\\n", OK_BEV_OFF, OK_BEV_WALL, OK_BEV_LANE);', "  return 0;", "}"]
    src.write_text("\n".join(lines) + "\n")
    exe = tmp_path / "layout"
    subprocess.run(["g++", "-x", "c++", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert got[0] == C.sizeof(_capi.OkBevQuery)
    assert got[1:-3] == [getattr(_capi.OkBevQuery, f).offset for f in FIELDS]
    assert got[-3:] == [ok.BEV_OFF, ok.BEV_WALL, ok.BEV_LANE]


def test_no_device_means_no_bev_query():
    with ok.Env(device=-1) as e:
        e.add_named_track("Monza")
        x = np.array([100.0, 200.0], dtype=np.float32)
        out = np.empty((2, 8, 8), dtype=np.uint8)
        with pytest.raises(ok.OkError) as ex:
            e.bev_query(x, x, x, 8, 8, 1.0)
        assert ex.value.code == _capi.OK_ERR_NO_DEVICE
        with pytest.raises(ok.OkError) as ex:
            e.bev_query_device(x.ctypes.data, x.ctypes.data, x.ctypes.data, 2, 8, 8, 1.0, out.ctypes.data)
        assert ex.value.code == _capi.OK_ERR_NO_DEVICE


BAD_IMAGES = [dict(height=0), dict(height=1025), dict(width=0), dict(width=1025), dict(scale=0.0), dict(scale=-1.0),
              dict(scale=float("nan")), dict(scale=float("inf")), dict(scale=1e39), dict(ahead=float("nan")),
              dict(ahead=float("inf")), dict(ahead=-float("inf"))]


def _image(**bad):
    a = dict(height=8, width=8, scale=1.0, ahead=0.0)
    a.update(bad)
    return a


@pytest.mark.parametrize("bad", BAD_IMAGES, ids=lambda b: "-".join(f"{k}={v}" for k, v in b.items()))
def test_env_bev_rejects_bad_images_before_the_library(bad):
    with ok.Env(device=-1) as e:  # the library would answer OK_ERR_NO_DEVICE: a ValueError comes from the wrapper
        e.add_named_track("Monza")
        a = np.zeros(3, dtype=np.float32)
        with pytest.raises(ValueError):
            e.bev_query(a, a, a, **_image(**bad))
        with pytest.raises(ValueError):
            e.bev_query_device(a.ctypes.data, a.ctypes.data, a.ctypes.data, 3, d_out=a.ctypes.data, **_image(**bad))


def test_env_bev_rejects_bad_poses_before_the_library():
    with ok.Env(device=-1) as e:
        e.add_named_track("Monza")
        a3, a4 = np.zeros(3, dtype=np.float32), np.zeros(4, dtype=np.float32)
        p = a3.ctypes.data
        for args in ((a3, a4, a3), (a3, a3, a4), (a4, a3, a3), (np.zeros((2, 2), dtype=np.float32),) * 3):
            with pytest.raises(ValueError):
                e.bev_query(*args, 8, 8, 1.0)
        with pytest.raises(ValueError):
            e.bev_query(a3, a3, a3, 8, 8, 1.0, track_id=np.zeros(4, dtype=np.int32))
        for ptrs in ((None, p, p, p), (p, None, p, p), (p, p, None, p), (p, p, p, None), (0, p, p, p)):
            with pytest.raises(ValueError):
                e.bev_query_device(ptrs[0], ptrs[1], ptrs[2], 3, 8, 8, 1.0, ptrs[3])
        with pytest.raises(ValueError):
            e.bev_query_device(p, p, p, -1, 8, 8, 1.0, p)
    with ok.Env(device=-1) as e:  # no track
        a = np.zeros(3, dtype=np.float32)
        with pytest.raises(ValueError):
            e.bev_query(a, a, a, 8, 8, 1.0)
        with pytest.raises(ValueError):
            e.bev_query_device(a.ctypes.data, a.ctypes.data, a.ctypes.data, 3, 8, 8, 1.0, a.ctypes.data)


class _NoLibrary:
    def __getattr__(self, name):
        raise AssertionError(f"the library was called ({name}) although the arguments are malformed")


def test_batch_env_bev_rejects_bad_arguments_before_the_library():
    env = BatchEnv.__new__(BatchEnv)  # no device here: only what bev() reads before its first call
    env.env, env.device = _NoLibrary(), torch.device("cpu")
    a3, a4 = torch.zeros(3), torch.zeros(4)
    for bad in BAD_IMAGES:
        with pytest.raises(ValueError):
            env.bev(x=a3, y=a3, rot=a3, **_image(**bad))
    for args in ((a3, a4, a3), (a3, a3, a4), (a4, a3, a3), (torch.zeros(2, 2),) * 3):
        with pytest.raises(ValueError):
            env.bev(x=args[0], y=args[1], rot=args[2])
    with pytest.raises(ValueError):
        env.bev(x=a3, y=a3)
    with pytest.raises(ValueError):
        env.bev(x=a3, y=a3, rot=a3, track_id=torch.zeros(4, dtype=torch.int32))


def _even_odd_f64(loop, px, py):
    """the even-odd rule in float64, edges (i, j = i - 1 cyclic): for each edge, only the points with min y <= py < max y
    (the PNPOLY y test) are looked at, found by bisection in the points sorted by y"""
    p = loop.astype(np.float64)
    xi, yi = p[:, 0], p[:, 1]
    xj, yj = np.roll(xi, 1), np.roll(yi, 1)
    order = np.argsort(py, kind="stable")
    sy, sx = py[order], px[order]
    inside = np.zeros(len(px), dtype=bool)
    lo = np.searchsorted(sy, np.minimum(yi, yj), "left")
    hi = np.searchsorted(sy, np.maximum(yi, yj), "left")
    for e in np.nonzero(hi > lo)[0]:
        s = slice(lo[e], hi[e])
        x_cross = (xj[e] - xi[e]) * (sy[s] - yi[e]) / (yj[e] - yi[e]) + xi[e]
        inside[s] ^= sx[s] < x_cross
    out = np.empty_like(inside)
    out[order] = inside
    return out


def _edge_distance(loops, px, py):
    """float64 distance of each point to the nearest edge of the loops"""
    best = np.full(len(px), np.inf)
    for loop in loops:
        p = loop.astype(np.float64)
        a, b = np.roll(p, 1, axis=0), p
        d = b - a
        for k in range(len(px)):
            q = np.array([px[k], py[k]])
            t = np.clip(((q - a) * d).sum(1) / np.maximum((d * d).sum(1), 1e-300), 0.0, 1.0)
            best[k] = min(best[k], float(np.sqrt((((a + t[:, None] * d) - q) ** 2).sum(1)).min()))
    return best


@pytest.mark.parametrize("name", ["Monza", "Spa", "Austin", "YasMarina"])
def test_oracle_matches_a_float64_even_odd_rule(name):
    ora = BevOracle()
    ora.add_track(ok.track_columns(name))
    rng = np.random.default_rng(sum(map(ord, name)))
    cx, cy = ora.track_array(0, "x"), ora.track_array(0, "y")
    n = 100_000
    i = rng.integers(0, len(cx), n)
    px = (cx[i] + rng.normal(0.0, 15.0, n)).astype(np.float32)
    py = (cy[i] + rng.normal(0.0, 15.0, n)).astype(np.float32)
    got = ora.bev(0, px, py, np.zeros(n, np.float32), 1, 1, 1.0)[:, 0, 0]  # a 1x1 image samples the pose itself
    loops = [ora.track_array(0, nm) for nm in LOOPS]
    k = sum(_even_odd_f64(lp, px.astype(np.float64), py.astype(np.float64)).astype(np.int32) for lp in loops)
    want = np.where(k == 2, ok.BEV_LANE, np.where(k % 2 == 1, ok.BEV_WALL, ok.BEV_OFF)).astype(np.uint8)
    assert set(np.unique(k)) >= {0, 1, 2}, np.unique(k)
    bad = np.nonzero(got != want)[0]
    assert len(bad) <= 10, len(bad)
    d = _edge_distance(loops, px[bad].astype(np.float64), py[bad].astype(np.float64))
    assert (d < 1e-3).all(), d
    ora.close()


def test_every_centre_line_point_is_lane():
    ora = BevOracle()
    for t, nm in enumerate(ok.track_names()):
        ora.add_track(ok.track_columns(nm))
        cx, cy = ora.track_array(t, "x"), ora.track_array(t, "y")
        got = ora.bev(t, cx, cy, np.zeros(len(cx), np.float32), 1, 1, 1.0)
        assert (got == ok.BEV_LANE).all(), (nm, np.nonzero(got.ravel() != ok.BEV_LANE)[0][:5])
    ora.close()

"""CPU: the host beam-table builder at table geometries other than the default 2 px x 256 bins.  A synthetic track folded
tightly enough that a 64 px cell reaches more than 1,024 wall segments, where the builder cuts a list at 4 + 4 * 255
candidates and lowers its completeness distance below the first candidate it leaves out; and a geometry whose table
cannot be addressed, which must fail before any list is built.  tests/test_gpu_beam_geometry.py runs the kernels on
these tables."""
import math

import numpy as np
import pytest

import openkitchen_b200 as ok

MAX_LIST = 4 + 4 * 255  # kBeamInline + 4 * kBeamMaxRest (ok_beam.hpp)
CELL_MARGIN, ANGLE_MARGIN = 0.0625, 1e-4  # kBeamCellMargin, kBeamAngleMargin (ok_beam.hpp)
FOLD_POINTS = 1200  # centre-line points 0 .. FOLD_POINTS - 1 are the folded stretch


def folded_track():
    """A circle of radius 1,000 (raw units) whose first stretch is a zig-zag of FOLD_POINTS points, 6 raw units to each side
    of its axis and 0.3 apart along it: after the fit to the window about 1,200 points, 4,800 wall segments, lie within
    230 px.  5,248 segments in all, a track blob that still fits the kernels' shared memory."""
    th = np.linspace(0.0, 2.0 * np.pi, 120, endpoint=False)[8:]
    k = np.arange(FOLD_POINTS)
    ph = (k % 40) / 20.0
    x = np.concatenate([1000.0 + 10.0 * np.where(ph < 1.0, 2.0 * ph - 1.0, 3.0 - 2.0 * ph), 1000.0 * np.cos(th)])
    y = np.concatenate([-60.0 + 0.3 * k, 1000.0 * np.sin(th)])
    w = np.full(len(x), 4.0)
    return tuple(np.asarray(c, np.float32) for c in (x, y, w, w))


# ---- the builder's exact list distance, restated in binary64 (ok_beam_geom.hpp, Builder::build_row) ----------------
def _cross(a, b):
    return a[0] * b[1] - a[1] * b[0]


def _hull8(pts):
    pts = sorted(pts)
    out = []
    for p in pts:
        while len(out) >= 2 and _cross((out[-1][0] - out[-2][0], out[-1][1] - out[-2][1]), (p[0] - out[-2][0], p[1] - out[-2][1])) <= 0:
            out.pop()
        out.append(p)
    lo = len(out) + 1
    for p in reversed(pts[:-1]):
        while len(out) >= lo and _cross((out[-1][0] - out[-2][0], out[-1][1] - out[-2][1]), (p[0] - out[-2][0], p[1] - out[-2][1])) <= 0:
            out.pop()
        out.append(p)
    return out[:-1] if len(out) > 1 else out


def _clip(poly, n):
    out = []
    for i, a in enumerate(poly):
        b = poly[(i + 1) % len(poly)]
        fa, fb = _cross(n, a), _cross(n, b)
        if fa >= 0:
            out.append(a)
        if (fa >= 0) != (fb >= 0):
            t = fa / (fa - fb)
            out.append((a[0] + t * (b[0] - a[0]), a[1] + t * (b[1] - a[1])))
    return out


def _origin_distance(poly):
    if not poly:
        return math.inf
    if len(poly) == 1:
        return math.hypot(*poly[0])
    inside, best = len(poly) >= 3, math.inf
    for i, a in enumerate(poly):
        b = poly[(i + 1) % len(poly)]
        e = (b[0] - a[0], b[1] - a[1])
        if _cross(e, (-a[0], -a[1])) < 0:
            inside = False
        l2 = e[0] * e[0] + e[1] * e[1]
        t = min(1.0, max(0.0, (-(a[0] * e[0]) - a[1] * e[1]) / l2 if l2 > 0 else 0.0))
        best = min(best, math.hypot(a[0] + t * e[0], a[1] + t * e[1]))
    return 0.0 if inside else best


def list_distances(seg, x0, y0, h, nb, ix, iy, b):
    """dist(C, b, S) of every segment (ok_beam.hpp): the origin's distance to (S (+) -C) clipped to the bin's widened cone,
    C the cell grown by the margin; inf where the clipped set is empty"""
    bx0, bx1 = x0 + ix * h - CELL_MARGIN, x0 + (ix + 1) * h + CELL_MARGIN
    by0, by1 = y0 + iy * h - CELL_MARGIN, y0 + (iy + 1) * h + CELL_MARGIN
    dbin = 2.0 * math.pi / nb
    lo = (math.cos(b * dbin - ANGLE_MARGIN), math.sin(b * dbin - ANGLE_MARGIN))
    hi = (math.cos((b + 1) * dbin + ANGLE_MARGIN), math.sin((b + 1) * dbin + ANGLE_MARGIN))
    out = np.full(len(seg), np.inf)
    for s, g in enumerate(seg.astype(np.float64)):
        pts = [(g[2 * e] - (bx1 if k & 1 else bx0), g[2 * e + 1] - (by1 if k & 2 else by0)) for e in range(2) for k in range(4)]
        out[s] = _origin_distance(_clip(_clip(_hull8(pts), lo), (-hi[0], -hi[1])))
    return out


def truncated_entries(env, t, pts, rng, n_rays=400):
    """(point, angle) of rays from the given centre-line points whose list the builder cut at MAX_LIST candidates, with
    their lookups"""
    x, y = env.track_array(t, "x"), env.track_array(t, "y")
    found = []
    for _ in range(n_rays):
        i = int(rng.choice(pts))
        ang = float(np.float32(rng.uniform(-math.pi, math.pi)))
        got = env.beam_lookup_ex(t, float(x[i]), float(y[i]), ang)
        if got is not None and len(got[0]) == MAX_LIST:
            found.append((i, ang, got))
    return found


def test_folded_track_cuts_lists_below_the_first_omitted_candidate():
    """At 64 px x 8 bins the folded stretch gives lists of more than 1,024 candidates.  Such a list keeps exactly its
    1,024 nearest candidates (4 inline, 255 full rest chunks), in order, and its completeness distance d is lowered to
    below the distance of the first candidate it leaves out (by the builder's 1e-3 px and at most the 1/16 px
    quantisation).  With d left at the sampled completeness distance the kernels would trust a list that misses walls."""
    env = ok.Env(device=-1, beam_cell=64.0, beam_bins=8)
    t = env.add_track(folded_track())
    seg = env.track_array(t, "segments")
    assert len(seg) < 65535
    found = truncated_entries(env, t, np.arange(FOLD_POINTS), np.random.default_rng(5))
    assert len(found) > 100, "the folded stretch should cut most of its lists"
    lowered = [f for f in found if f[2][1] > 0.0]
    assert len(lowered) >= 5, "no cut list with a completeness distance above 0"
    x0, y0, h, nb = math.floor(float(seg[:, 0::2].min()) - 1.0), math.floor(float(seg[:, 1::2].min()) - 1.0), 64.0, 8
    checked = set()
    for i, ang, (items, d, d1, n_inline) in lowered:
        xi, yi = float(env.track_array(t, "x")[i]), float(env.track_array(t, "y")[i])
        ix, iy = int(np.float32(xi - np.float32(x0)) * np.float32(1.0 / h)), int(np.float32(yi - np.float32(y0)) * np.float32(1.0 / h))
        b = int(math.floor(np.float32(ang) * np.float32(nb / (2.0 * math.pi)))) & (nb - 1)
        if (ix, iy, b) in checked:
            continue
        checked.add((ix, iy, b))
        assert n_inline == 4 and len(set(items.tolist())) == MAX_LIST
        dist = list_distances(seg, x0, y0, h, nb, ix, iy, b).astype(np.float32)
        order = np.lexsort((np.arange(len(seg)), dist))  # the builder's (distance, segment) order
        assert items.tolist() == order[:MAX_LIST].tolist(), f"cell {(ix, iy)} bin {b}: not the 1,024 nearest candidates"
        omitted = float(dist[order[MAX_LIST]])
        assert d < omitted and d >= omitted - 1e-3 - 1.0 / 16, (d, omitted)
        if len(checked) == 3:
            break
    assert len(checked) == 3


def test_geometry_too_large_fails_before_building():
    """1 px x 1,024 bins passes the config check, but Zandvoort's rows and entries alone pass the table's 32-bit offsets:
    the build fails with OK_ERR_INVALID_ARG and "beam table too large" (before any list is built), and the env still
    builds a table of a geometry that fits"""
    env = ok.Env(device=-1, beam_cell=1.0, beam_bins=1024)
    with pytest.raises(ok.OkError) as err:
        env.beam_table_bytes(env.add_named_track("Zandvoort"))
    assert err.value.code == -1 and "beam table too large" in str(err.value)  # OK_ERR_INVALID_ARG
    small = ok.Env(device=-1, beam_cell=16.0, beam_bins=16)
    assert small.beam_table_bytes(small.add_named_track("Zandvoort")) > 0

"""CPU: races (OkRaces, include/openkitchen_b200.h).  The structs' layout against the C compiler, the entry points' refusal
without a device, the argument checks of the C entry point and of the wrappers, and the test-side restatement of the pass
(tests/race_oracle.py) against an independent float64 statement of what it computes: every car hit lies on the body's
circle, no opponent is nearer along the ray than the one reported, no ray misses a nearer car, and contact is exactly the
overlap set."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

import openkitchen_b200 as ok
from openkitchen_b200 import _capi
from oracle.api import Oracle
from tests.race_oracle import CONTACT, SENSE, Races, pack_races

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_struct_layout_matches_the_c_compiler(tmp_path):
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "openkitchen_b200.h"\n'
                   'int main(void) { printf("%zu %zu %zu %zu %zu %zu %zu %d %d", sizeof(OkRaces), offsetof(OkRaces, group), '
                   'offsetof(OkRaces, flags), offsetof(OkRaces, radius), sizeof(OkRaceBuffers), '
                   'offsetof(OkRaceBuffers, hit_car), offsetof(OkRaceBuffers, contact), OK_RACE_SENSE, OK_RACE_CONTACT); '
                   'return 0; }\n')
    exe = tmp_path / "layout"
    subprocess.run(["g++", "-x", "c++", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    v = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    R, B = _capi.OkRaces, _capi.OkRaceBuffers
    assert v == [C.sizeof(R), R.group.offset, R.flags.offset, R.radius.offset, C.sizeof(B), B.hit_car.offset,
                 B.contact.offset, _capi.RACE_SENSE, _capi.RACE_CONTACT]
    assert (SENSE, CONTACT) == (_capi.RACE_SENSE, _capi.RACE_CONTACT)


def test_every_entry_point_needs_a_device():
    lib = _capi.load()
    with ok.Env(device=-1) as e:
        e.add_named_track("Monza")
        races, bufs = _capi.OkRaces(group=8, flags=3, radius=4.0), _capi.OkRaceBuffers()
        for rc in (lib.ok_set_races(e.h, C.byref(races)), lib.ok_set_races(e.h, None),
                   lib.ok_get_races(e.h, C.byref(races)), lib.ok_race_buffers(e.h, C.byref(bufs))):
            assert rc == _capi.OK_ERR_NO_DEVICE
        for call in (lambda: e.set_races(8, 4.0), lambda: e.set_races(0), e.races, e.race_buffers_info):
            with pytest.raises(ok.OkError) as ex:
                call()
            assert ex.value.code == _capi.OK_ERR_NO_DEVICE
    assert lib.ok_set_races(None, None) == _capi.OK_ERR_INVALID_ARG


BAD = [(1, 3, 4.0), (-2, 3, 4.0), (1025, 3, 4.0), (8, 0, 4.0), (8, 4, 4.0), (8, 7, 4.0), (8, -1, 4.0), (8, 3, 0.0),
       (8, 3, -1.0), (8, 3, float("nan")), (8, 3, float("inf"))]


@pytest.mark.parametrize("group,flags,radius", BAD)
def test_bad_arguments_are_refused(group, flags, radius):
    """the C entry point checks its arguments before it asks for a device; the wrapper refuses the same ones"""
    lib = _capi.load()
    with ok.Env(device=-1) as e:
        r = _capi.OkRaces(group=group, flags=flags, radius=radius)
        assert lib.ok_set_races(e.h, C.byref(r)) == _capi.OK_ERR_INVALID_ARG
        if flags in (1, 2, 3):
            with pytest.raises(ValueError):
                e.set_races(group, radius, sense=bool(flags & 1), contact=bool(flags & 2))
    with ok.Env(device=-1) as e:
        with pytest.raises(ValueError):
            e.set_races(8, 4.0, sense=False, contact=False)


def test_off_ignores_the_other_fields():
    lib = _capi.load()
    with ok.Env(device=-1) as e:
        assert lib.ok_set_races(e.h, C.byref(_capi.OkRaces(group=0, flags=99, radius=-1.0))) == _capi.OK_ERR_NO_DEVICE


# ---- the restatement against a float64 rule ---------------------------------------------------------------------------
RADIUS = 4.0


def race_oracle(n=64, rays=16, group=8, mixed=True, seed=0, flags=SENSE | CONTACT, offset=0.0):
    """an oracle with the cars of each race packed along the first car's heading at random spacings (overlapping, in the
    lidar's crash band, in range and out of range), on two tracks (interleaved: races that mix tracks)"""
    ora = Oracle("port", reward_mode=ok.REWARD_CONSTANT, sensor_offset=offset)
    for nm in ("Monza", "Spa"):
        ora.add_track(ok.track_columns(nm))
    fan = ok.ray_fan(rays)
    tid = (np.arange(n) % 2 if mixed else np.arange(n) * 2 // n).astype(np.int32)
    ora.alloc_agents(n, fan, tid)
    pts = np.array([(i * 2654435761 % 2**32) % ora.track_points(int(tid[i])) for i in range(n)], dtype=np.int32)
    ora.reset(None, pts)
    px, py, pr = pack_races(ora.buffer("pos_x"), ora.buffer("pos_y"), ora.buffer("rot"), tid, group, np.random.default_rng(seed))
    ora.buffer("pos_x")[:], ora.buffer("pos_y")[:], ora.buffer("rot")[:] = px, py, pr
    ora.cast_rays()
    return ora, Races(ora, fan, group, RADIUS, flags)


def t64(o, d, c, r, limit):
    """the exact first parameter at which the ray o + t d (t >= 0) meets the disc of radius r around c, in float64; 0 when
    o is inside; inf when it misses or meets it beyond `limit`"""
    w = c - o
    a, b, cc = d @ d, w @ d, w @ w - r * r
    if cc <= 0:
        return 0.0
    disc = b * b - a * cc
    if b <= 0 or disc < 0:
        return math.inf
    t = (b - math.sqrt(disc)) / a
    return t if t <= limit else math.inf


@pytest.mark.parametrize("group,mixed,offset", [(2, False, 0.0), (7, True, 0.0), (8, True, 3.0), (32, False, 0.0)])
def test_restatement_against_a_float64_rule(group, mixed, offset):
    ora, races = race_oracle(n=70, group=group, mixed=mixed, seed=group, offset=offset)
    rng_ = float(ora.cfg.sensor_range)
    before = {k: ora.buffer(k).copy() for k in ("crashed", "hit_t", "hit_abs")}
    races.apply()
    live = np.flatnonzero(before["crashed"] == 0)
    x, y = ora.buffer("pos_x").astype(np.float64), ora.buffer("pos_y").astype(np.float64)
    hit_t, hit_abs, hit_car = ora.buffer("hit_t"), ora.buffer("hit_abs"), races.hit_car
    margin = 1e-3 * (rng_ + RADIUS)  # px: far above the binary32 rounding of the test, far below the car's size
    hits = 0
    for i in live:
        opp = races.opponents(int(i))
        ox, oy, _, _, dx, dy = races.rays(int(i))
        o = np.array([ox, oy], dtype=np.float64)
        for r in range(ora.rays):
            d = np.array([dx[r], dy[r]], dtype=np.float64)
            ts = np.array([t64(o, d, np.array([x[j], y[j]]), RADIUS, rng_) for j in opp]) if opp.size else np.zeros(0)
            j = hit_car[i, r]
            if j >= 0:
                hits += 1
                assert j in opp
                t = float(hit_t[i, r])
                assert t < before["hit_t"][i, r] and ora.buffer("hit_seg")[i, r] == -1
                dist = math.hypot(float(hit_abs[i, r, 0]) - x[j], float(hit_abs[i, r, 1]) - y[j])
                if t > 0:
                    assert abs(dist - RADIUS) <= 1e-3 * (RADIUS + t), (i, r, j, dist)  # on the circle
                else:
                    assert dist <= RADIUS + 1e-3  # the origin is inside the body
                assert ts.min() >= t - margin, (i, r, t, ts.min())  # no opponent nearer along the ray
            else:
                limit = min(float(before["hit_t"][i, r]), rng_)
                assert not np.any(ts < limit - margin), (i, r)  # no nearer car was missed
    assert hits > 0
    # contact: exactly the overlap set, in float64
    crashed_by_contact = np.zeros(ora.n, dtype=bool)
    for i in live:
        opp = races.opponents(int(i))
        crashed_by_contact[i] = bool(np.any(np.hypot(x[i] - x[opp], y[i] - y[opp]) < 2 * RADIUS))
    assert crashed_by_contact.any()
    ora2, races2 = race_oracle(n=70, group=group, mixed=mixed, seed=group, flags=CONTACT, offset=offset)
    races2.apply()
    assert np.array_equal(races2.contact.astype(bool), crashed_by_contact)
    assert np.all(races.contact.astype(bool) >= crashed_by_contact)  # sense can only add crashes
    assert np.all(races2.hit_car == -1)  # contact only: the lidar does not see cars


def test_crashed_agents_are_left_alone():
    ora, races = race_oracle(n=40, group=8, seed=3)
    ora.buffer("crashed")[::3] = 1
    snap = {k: ora.buffer(k).copy() for k in ("hit_t", "hit_abs", "min_dist2", "done")}
    races.apply()
    idx = np.arange(0, 40, 3)
    assert np.all(races.contact[idx] == 0) and np.all(races.hit_car[idx] == -1)
    for k, v in snap.items():
        assert np.array_equal(ora.buffer(k)[idx].view(np.uint8), v[idx].view(np.uint8)), k


def test_nan_poses_neither_hit_nor_are_hit():
    ora, races = race_oracle(n=32, group=8, seed=4)
    ora.buffer("pos_x")[[1, 9]] = np.nan
    races.apply()
    assert np.all(races.hit_car[[1, 9]] == -1) and races.contact[1] == 0 and races.contact[9] == 0
    assert not np.isin(races.hit_car, [1, 9]).any()

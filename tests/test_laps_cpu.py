"""CPU: lap accounting (OkLaps, include/openkitchen_b200.h).  The structs' layout against the C compiler, the entry points'
refusal without a device, the wrappers' argument checks, and the test-side restatement of the tick rule
(tests/laps_oracle.py): the vectorised rule against a one-agent-at-a-time statement of the header's definition, and the
accounting over the port oracle."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import openkitchen_b200 as ok
from openkitchen_b200 import _capi
from oracle.api import Oracle
from tests.laps_oracle import FIELDS, Laps, lap_rule

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_struct_layout_matches_the_c_compiler(tmp_path):
    fields = [f for f, _ in _capi.OkLapBuffers._fields_]
    src = tmp_path / "layout.c"
    offs = " ".join(f'printf("%zu ", offsetof(OkLapBuffers, {f}));' for f in fields)
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "openkitchen_b200.h"\n'
                   'int main(void) { printf("%zu %zu %zu %zu ", sizeof(OkLaps), offsetof(OkLaps, enabled), '
                   f'offsetof(OkLaps, target), sizeof(OkLapBuffers)); {offs} return 0; }}\n')
    exe = tmp_path / "layout"
    subprocess.run(["g++", "-x", "c++", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    v = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert v[0] == C.sizeof(_capi.OkLaps) and v[1] == _capi.OkLaps.enabled.offset and v[2] == _capi.OkLaps.target.offset
    assert v[3] == C.sizeof(_capi.OkLapBuffers)
    assert v[4:] == [getattr(_capi.OkLapBuffers, f).offset for f in fields]
    assert fields == list(_capi.LAP_ARRAYS) == list(FIELDS)


def test_every_entry_point_needs_a_device():
    lib = _capi.load()
    with ok.Env(device=-1) as e:
        e.add_named_track("Monza")
        laps, bufs = _capi.OkLaps(enabled=1, target=2), _capi.OkLapBuffers()
        for rc in (lib.ok_set_laps(e.h, C.byref(laps), None), lib.ok_set_laps(e.h, None, None),
                   lib.ok_get_laps(e.h, C.byref(laps)), lib.ok_lap_buffers(e.h, C.byref(bufs))):
            assert rc == _capi.OK_ERR_NO_DEVICE
        for call in (lambda: e.set_laps(1), e.laps, e.lap_buffers_info):
            with pytest.raises(ok.OkError) as ex:
                call()
            assert ex.value.code == _capi.OK_ERR_NO_DEVICE
    assert lib.ok_set_laps(None, None, None) == _capi.OK_ERR_INVALID_ARG


def test_wrappers_reject_bad_arguments():
    with ok.Env(device=-1) as e:
        with pytest.raises(ValueError):
            e.set_laps(-1)
        with pytest.raises(ValueError):
            e.set_laps(-5, enabled=False)


def _scalar_rule(s, n, P, target):
    """the header's rule 2 for one agent, in Python integers"""
    def i32(v):
        return (v + 2**31) % 2**32 - 2**31

    s = dict(s)
    d = i32(n - s["lap_idx"])
    if 2 * d > P:
        d -= P
    elif 2 * d <= -P:
        d += P
    s["progress"] = i32(s["progress"] + d)
    s["lap_idx"] = n
    s["ticks"] = (s["ticks"] + 1) % 2**32
    if s["progress"] >= (s["laps"] + 1) * P:
        s["laps"] = i32(s["laps"] + 1)
        s["last_lap"] = (s["ticks"] - s["lap_start"]) % 2**32
        s["lap_start"] = s["ticks"]
    if target > 0 and s["laps"] >= target:
        s["completed"] = 1
    return s


def _check(s, n, P, target, moved):
    got = lap_rule(s, n, P, target, moved)
    Ps = np.broadcast_to(np.asarray(P), moved.shape)
    for a in range(len(moved)):
        one = {f: int(s[f][a]) for f in FIELDS}
        want = _scalar_rule(one, int(n[a]), int(Ps[a]), target) if moved[a] else one
        for f in FIELDS:
            assert int(got[f][a]) == want[f], (f, a, one, int(n[a]), int(Ps[a]))
        assert got[f].dtype == FIELDS[f]
    return got


@pytest.mark.parametrize("P", [7, 8, 739, 740, 2000, 2001])
def test_rule_equals_the_definition(P):
    rng = np.random.default_rng(P)
    m = 4000
    s = {"lap_idx": rng.integers(0, P, m).astype(np.int32), "progress": rng.integers(-3 * P, 3 * P, m).astype(np.int32),
         "laps": rng.integers(0, 3, m).astype(np.int32), "ticks": rng.integers(0, 2**32, m, dtype=np.uint64).astype(np.uint32),
         "lap_start": rng.integers(0, 2**32, m, dtype=np.uint64).astype(np.uint32),
         "last_lap": rng.integers(0, 1000, m).astype(np.uint32), "completed": rng.integers(0, 2, m).astype(np.uint8)}
    # d exactly +-P/2 (and the neighbours) on a slice, arbitrary indices on the rest
    n = rng.integers(0, P, m)
    half = np.arange(m) < 600
    off = np.array([P // 2, -(P // 2), (P + 1) // 2, -((P + 1) // 2), P // 2 + 1, -(P // 2) - 1])
    n[half] = (s["lap_idx"][half] + off[np.arange(half.sum()) % off.size]) % P
    # progress just below a lap boundary, and at the 32-bit limits
    s["progress"][600:900] = ((s["laps"][600:900].astype(np.int64) + 1) * P - rng.integers(0, 4, 300)).astype(np.int32)
    s["progress"][900:950] = np.int32(2**31 - 1) - rng.integers(0, P, 50).astype(np.int32)
    s["progress"][950:1000] = np.int32(-(2**31)) + rng.integers(0, P, 50).astype(np.int32)
    s["laps"][900:1000] = np.int32(2**31 - 1)
    moved = rng.random(m) < 0.8
    for target in (0, 1, 3):
        _check(s, n, P, target, moved)


def test_reversal_across_a_lap_boundary_counts_the_lap_once():
    """drive to one point short of a lap, across it (a lap), back across it, and forward again: the lap is counted once,
    and counted again only once progress passes the next multiple of P"""
    P = 101
    s = {f: np.zeros(1, dt) for f, dt in FIELDS.items()}
    s["lap_idx"][0] = 10
    path = list(range(11, 101)) + list(range(0, 12)) + list(range(10, 5, -1)) + list(range(6, 15))
    seen = []
    for t, n in enumerate(path):
        s = _check(s, np.array([n]), P, 2, np.array([True]))
        seen.append((int(s["progress"][0]), int(s["laps"][0])))
    assert seen[99] == (P - 1, 0) and seen[100] == (P, 1)  # back at index 10: the first lap
    assert int(s["last_lap"][0]) == 101 and int(s["completed"][0]) == 0
    assert seen[106] == (P - 4, 1) and max(l for _, l in seen) == 1  # the reversal lowers progress, not laps
    assert seen[-1] == (P + 4, 1)


def _oracle(n=24, auto_reset=1, reward=ok.REWARD_CONSTANT):
    ora = Oracle("port", auto_reset=auto_reset, reward_mode=reward)
    for nm in ("Monza", "Spa"):
        ora.add_track(ok.track_columns(nm))
    ora.alloc_agents(n, ok.ray_fan(9), (np.arange(n) % 2).astype(np.int32))
    return ora


def test_completed_agents_are_auto_reset_and_restart():
    laps = Laps(_oracle())
    laps.set(True, 1)
    laps.s["progress"][:12] = (laps.n_points[:12] - 2).astype(np.int32)
    done_seen = reset_seen = 0
    for step in range(60):
        laps.ora.fill_random_actions(step)
        before = laps.s["completed"].copy()
        laps.step()
        done = laps.ora.buffer("done")
        assert np.array_equal(done, (laps.ora.buffer("crashed") | laps.s["completed"]).astype(np.uint8))
        done_seen += int(laps.s["completed"].sum())
        # a completed agent restarts at the next tick: one tick of progress from its new point
        reset_seen += int(np.sum(before.astype(bool) & (laps.s["ticks"] == 1)))
    assert done_seen > 0 and reset_seen > 0


def test_accounting_off_leaves_the_oracle_as_it_is():
    a, b = _oracle(), Laps(_oracle())
    for step in range(80):
        a.fill_random_actions(step)
        a.step()
        b.ora.fill_random_actions(step)
        b.step()
    for name in ("pos_x", "rot", "done", "nearest_idx", "reset_pt", "obs"):
        assert np.array_equal(a.buffer(name).view(np.uint8), b.ora.buffer(name).view(np.uint8)), name

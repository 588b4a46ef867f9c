"""CPU: reset draws (OkResetDraws, include/openkitchen_b200.h).  The struct's layout against the C compiler, the entry
points' refusal without a device, the Python wrappers' argument checks, and the test-side restatement of the header's
definition (tests/reset_draws_oracle.py): its Philox against the oracle's, its mapping against a scalar statement of the
definition, the distribution, the alternating sign, and sharding with drawn auto-resets over the port oracle."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from scipy import stats

import openkitchen_b200 as ok
from openkitchen_b200 import _capi
from oracle.api import Oracle
from tests.reset_draws_oracle import DrawnResets, draw, philox4x32_10

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_struct_layout_matches_the_c_compiler(tmp_path):
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "openkitchen_b200.h"\n'
                   'int main(void) { printf("%zu %zu %zu %d %d %d\\n", sizeof(OkResetDraws), offsetof(OkResetDraws, seed), '
                   'offsetof(OkResetDraws, flags), OK_RESET_DRAW_POINT, OK_RESET_DRAW_LANE, OK_RESET_DRAW_HEADING); return 0; }\n')
    exe = tmp_path / "layout"
    subprocess.run(["g++", "-x", "c++", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    size, o_seed, o_flags, p, l, h = (int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split())
    assert size == C.sizeof(_capi.OkResetDraws)
    assert o_seed == _capi.OkResetDraws.seed.offset and o_flags == _capi.OkResetDraws.flags.offset
    assert (p, l, h) == (ok.RESET_DRAW_POINT, ok.RESET_DRAW_LANE, ok.RESET_DRAW_HEADING) == (1, 2, 4)


def test_every_entry_point_needs_a_device():
    lib = _capi.load()
    with ok.Env(device=-1) as e:
        e.add_named_track("Monza")
        d = _capi.OkResetDraws(seed=1, flags=7)
        ptr = C.c_void_p()
        idx = np.zeros(1, dtype=np.int64)
        for rc in (lib.ok_set_reset_draws(e.h, C.byref(d)), lib.ok_get_reset_draws(e.h, C.byref(d)),
                   lib.ok_reset_agents_drawn(e.h, None, None, 4, None),
                   lib.ok_reset_agents_drawn_host(e.h, idx.ctypes.data_as(C.c_void_p), None, 1, None),
                   lib.ok_reset_draw_counts(e.h, C.byref(ptr))):
            assert rc == _capi.OK_ERR_NO_DEVICE
        for call in (lambda: e.set_reset_draws(1), e.reset_draws, lambda: e.reset_drawn(idx)):
            with pytest.raises(ok.OkError) as ex:
                call()
            assert ex.value.code == _capi.OK_ERR_NO_DEVICE


def test_wrappers_reject_bad_arguments():
    with ok.Env(device=-1) as e:
        e.add_named_track("Monza")
        e.n = 4  # what alloc_agents would have recorded: the checks below come before any call into the library
        with pytest.raises(ValueError):
            e.set_reset_draw_flags(1, 8)
        with pytest.raises(ValueError):
            e.set_reset_draw_flags(1, -1)
        with pytest.raises(ValueError):
            e.reset_drawn(agent_idx=[0, 1], mask=np.ones(4, np.uint8))
        with pytest.raises(ValueError):
            e.reset_drawn(mask=np.ones(3, np.uint8))
        with pytest.raises(ValueError):
            e.reset_drawn_device(d_agent_idx=1, d_mask=2, n=4)
        with pytest.raises(ValueError):
            e.reset_drawn_device(d_mask=2, n=3)
        with pytest.raises(ValueError):
            e.reset_drawn_device(n=5)
        with pytest.raises(ValueError):
            e.reset_drawn_device(d_agent_idx=1)


def test_draw_equals_the_definition():
    """10^5 (id, k) pairs, every flag combination: the vectorised draw against the definition stated one agent at a time,
    with the oracle's own Philox4x32-10 (oko_philox4x32_10) and integer arithmetic"""
    ora = Oracle("port")
    rng = np.random.default_rng(7)
    m = 100_000
    ids = rng.integers(0, 2**40, m, dtype=np.uint64)
    ids[:3] = [0, 2**32 - 1, 2**32]
    k = rng.integers(0, 2**32, m, dtype=np.uint64)
    n_pts = rng.integers(2, 3000, m)
    flags = np.arange(m) % 8
    seed = 0xC0FFEE
    o = np.array([ora.philox([int(i) & 0xFFFFFFFF, int(i) >> 32, int(kk), 0], [seed, 0x525354]) for i, kk in zip(ids, k)],
                 dtype=np.uint64)
    mine = philox4x32_10(ids & np.uint64(0xFFFFFFFF), ids >> np.uint64(32), k, 0, seed, 0x525354)
    for w in range(4):
        assert np.array_equal(mine[w], o[:, w]), w
    for f in range(8):
        sel = np.flatnonzero(flags == f)
        pt, alpha, off = draw(seed, f, ids[sel], k[sel], n_pts[sel], (n_pts[sel] - 1).astype(np.int32))
        for j, i in enumerate(sel[:2000]):
            o0, o1, o2 = (int(x) for x in o[i, :3])
            want_pt = (o0 * int(n_pts[i])) >> 32 if f & 1 else int(n_pts[i]) - 1
            want_alpha = np.float32(10 + ((o1 * 81) >> 32)) / np.float32(100)
            mag = float(45 + ((o2 * 46) >> 32))
            want_off = np.float32((mag if int(k[i]) & 1 else -mag) if f & 4 else 0.0)
            assert pt[j] == want_pt and alpha[j].view(np.uint32) == want_alpha.view(np.uint32), (f, i)
            assert off[j].view(np.uint32) == want_off.view(np.uint32), (f, i)


def test_draws_are_uniform():
    """10^6 draws: pt over P points, alpha over its 81 values, the offset's magnitude over its 46 values"""
    n = 1_000_000
    ids = np.arange(n, dtype=np.uint64) + np.uint64(12345)
    k = np.arange(n, dtype=np.uint64) % np.uint64(7)
    P = 677
    pt, alpha, off = draw(0x1234, 7, ids, k, P, 0)
    cnt = np.bincount(pt, minlength=P)
    assert cnt.size == P and stats.chisquare(cnt).pvalue > 1e-4
    a = np.rint(alpha.astype(np.float64) * 100).astype(np.int64)
    assert a.min() == 10 and a.max() == 90
    assert np.all(alpha == (a.astype(np.float32) / np.float32(100)))
    assert stats.chisquare(np.bincount(a - 10, minlength=81)).pvalue > 1e-4
    mag = np.abs(off).astype(np.int64)
    assert mag.min() == 45 and mag.max() == 90
    assert stats.chisquare(np.bincount(mag - 45, minlength=46)).pvalue > 1e-4


def test_sign_alternates_with_the_counter():
    for agent in (0, 5, 2**33 + 1):
        _, _, off = draw(9, 4, np.full(12, agent, np.uint64), np.arange(12, dtype=np.uint64), 100, 0)
        assert list(np.sign(off)) == [-1.0, 1.0] * 6
    # without HEADING the offset is zero, without POINT the given point
    pt, _, off = draw(9, 2, np.array([3], np.uint64), np.array([1], np.uint64), 100, 42)
    assert (int(pt[0]), float(off[0])) == (42, 0.0)


def _oracle(names, n, fan, tid, base=0):
    ora = Oracle("port", auto_reset=1, reward_mode=ok.REWARD_CMAES_PROGRESS, agent_id_base=base)
    for nm in names:
        ora.add_track(ok.track_columns(nm))
    ora.alloc_agents(n, fan, tid)
    return ora


def test_shard_reproduces_its_slice_with_drawn_auto_resets():
    names = ["Monza", "Spa", "Silverstone"]
    n, lo = 24, 10
    fan = ok.ray_fan(9)
    tid = (np.arange(n) % len(names)).astype(np.int32)
    full = DrawnResets(_oracle(names, n, fan, tid), 0xABCD, 7)
    shard = DrawnResets(_oracle(names, n - lo, fan, tid[lo:], base=lo), 0xABCD, 7)
    for step in range(150):
        for d in (full, shard):
            d.ora.fill_random_actions(step)
            d.step()
    assert full.k.sum() > n, "too few auto-resets for the test to mean anything"
    assert np.array_equal(full.k[lo:], shard.k)
    for name in ("pos_x", "pos_y", "rot", "reset_pt", "start_x", "start_y", "obs", "crashed", "prev_idx"):
        assert np.array_equal(full.ora.buffer(name)[lo:].view(np.uint8), shard.ora.buffer(name).view(np.uint8)), name


def test_draws_off_leave_the_oracle_as_it_is():
    """flags 0: the oracle's stride auto-reset, counters untouched; explicit drawn resets go to kStartingIdx and count"""
    names, fan = ["Monza"], ok.ray_fan(5)
    a = _oracle(names, 8, fan, None)
    b = DrawnResets(_oracle(names, 8, fan, None), 0x55, 0)
    for step in range(120):
        a.fill_random_actions(step)
        a.step()
        b.ora.fill_random_actions(step)
        b.step()
    for name in ("pos_x", "rot", "reset_pt", "obs"):
        assert np.array_equal(a.buffer(name).view(np.uint8), b.ora.buffer(name).view(np.uint8))
    assert not b.k.any()
    b.reset(mask=np.array([1, 0, 0, 1, 0, 0, 0, 0], np.uint8))
    assert list(b.k) == [1, 0, 0, 1, 0, 0, 0, 0]
    assert b.ora.buffer("reset_pt")[0] == 3 and b.ora.buffer("reset_pt")[3] == 3

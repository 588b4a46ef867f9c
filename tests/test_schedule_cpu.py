"""CPU: the tilings of the agent range (openkitchen_b200/csrc/ok_schedule.cpp), compiled with g++ next to a small C
wrapper and driven through ctypes.  Guided and balanced tilings must partition the agents into same-track tiles within
their caps; the cost-balanced tiling must minimise the slowest tile; the feedback model must ignore what carries no
information and damp what it learns."""
import ctypes as C
import itertools
import os
import subprocess

import numpy as np
import pytest

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "openkitchen_b200", "csrc")

WRAPPER = r'''
#include "ok_schedule.hpp"
#include <cstring>

namespace {
int64_t put(const std::vector<ok::Tile> &tiles, int64_t *out, int64_t cap)
{
    for (size_t i = 0; i < tiles.size() && static_cast<int64_t>(i) < cap; ++i)
        out[3 * i] = tiles[i].track, out[3 * i + 1] = tiles[i].count, out[3 * i + 2] = tiles[i].begin;
    return static_cast<int64_t>(tiles.size());
}
std::vector<ok::TileRun> runs_of(int64_t n_runs, const int32_t *track, const int64_t *begin, const int64_t *len, const int64_t *cap,
                                 const double *w)
{
    std::vector<ok::TileRun> runs;
    for (int64_t r = 0; r < n_runs; ++r)
        runs.push_back({track[r], begin[r], len[r], cap[r], w[r], 0});
    return runs;
}
} // namespace

extern "C" {
int64_t sch_guided(const int32_t *track_id, int64_t n, int big, int ctas, int tail_div, int64_t *out, int64_t cap)
{
    return put(ok::guided_tiles(track_id, n, big, ctas, tail_div), out, cap);
}

int64_t sch_balanced(const int32_t *track_id, int64_t n, int64_t max_tile, int ctas, int min_waves, int64_t *out, int64_t cap,
                     int64_t *target)
{
    std::vector<ok::TileRun> runs = ok::track_runs(track_id, n, max_tile);
    ok::BalancedTiling       bt   = ok::balanced_tiles(runs, max_tile, ctas, min_waves);
    *target                       = bt.target;
    return put(bt.tiles, out, cap);
}

int64_t sch_cost_balanced(int64_t n_runs, const int32_t *track, const int64_t *begin, const int64_t *len, const int64_t *cap,
                          const double *w, int64_t target, double c0, int64_t *out, int64_t out_cap, float *slowest_over_mean)
{
    std::vector<ok::TileRun> runs = runs_of(n_runs, track, begin, len, cap, w);
    return put(ok::cost_balanced_tiles(runs, target, c0, slowest_over_mean), out, out_cap);
}

// w: in / out.  Returns the number of re-cut tiles, or -1 for "no change".
int64_t sch_reweigh(int64_t n_runs, const int32_t *track, const int64_t *begin, const int64_t *len, const int64_t *cap, double *w,
                    int64_t n_tiles, const int64_t *tiles, const uint32_t *ns, int32_t *weighted, int64_t target, int64_t *out,
                    int64_t out_cap, float *balance)
{
    std::vector<ok::TileRun> runs = runs_of(n_runs, track, begin, len, cap, w);
    std::vector<ok::Tile>    cur;
    for (int64_t i = 0; i < n_tiles; ++i)
        cur.push_back({static_cast<int32_t>(tiles[3 * i]), static_cast<int32_t>(tiles[3 * i + 1]), tiles[3 * i + 2]});
    bool           wt      = *weighted != 0;
    ok::Reweighing rw;
    const bool     changed = ok::reweigh_runs(runs, cur, ns, wt, target, rw);
    *weighted              = wt;
    for (int64_t r = 0; r < n_runs; ++r)
        w[r] = runs[r].w;
    if (!changed)
        return -1;
    balance[0] = rw.balance_before, balance[1] = rw.balance_after;
    return put(rw.tiles, out, out_cap);
}
}
'''

_P = C.c_void_p


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    d = tmp_path_factory.mktemp("schedule")
    (d / "wrap.cpp").write_text(WRAPPER)
    so = d / "libschedule.so"
    subprocess.run(["/usr/bin/g++", "-std=c++17", "-O2", "-Wall", "-shared", "-fPIC", "-I", CSRC, "-o", str(so),
                    str(d / "wrap.cpp"), os.path.join(CSRC, "ok_schedule.cpp")], check=True)
    L = C.CDLL(str(so))
    L.sch_guided.restype = L.sch_balanced.restype = L.sch_cost_balanced.restype = L.sch_reweigh.restype = C.c_int64
    L.sch_guided.argtypes = [_P, C.c_int64, C.c_int, C.c_int, C.c_int, _P, C.c_int64]
    L.sch_balanced.argtypes = [_P, C.c_int64, C.c_int64, C.c_int, C.c_int, _P, C.c_int64, _P]
    L.sch_cost_balanced.argtypes = [C.c_int64, _P, _P, _P, _P, _P, C.c_int64, C.c_double, _P, C.c_int64, _P]
    L.sch_reweigh.argtypes = [C.c_int64, _P, _P, _P, _P, _P, C.c_int64, _P, _P, _P, C.c_int64, _P, C.c_int64, _P]
    return L


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def guided(lib, tid, big, ctas, tail_div):
    out = np.zeros((len(tid), 3), np.int64)
    k = lib.sch_guided(_p(tid), len(tid), big, ctas, tail_div, _p(out), len(tid))
    return out[:k]


def balanced(lib, tid, max_tile, ctas, waves):
    out, target = np.zeros((len(tid), 3), np.int64), np.zeros(1, np.int64)
    k = lib.sch_balanced(_p(tid), len(tid), max_tile, ctas, waves, _p(out), len(tid), _p(target))
    return out[:k], int(target[0])


class Runs:
    def __init__(self, lens, cap, w=None, tracks=None):
        lens = np.asarray(lens, np.int64)
        self.track = np.asarray(tracks if tracks is not None else np.arange(len(lens)), np.int32)
        self.begin = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.int64)
        self.len = lens
        self.cap = np.broadcast_to(np.asarray(cap, np.int64), lens.shape).copy()
        self.w = np.asarray(w if w is not None else np.ones(len(lens)), np.float64).copy()

    def args(self):
        return [len(self.len), _p(self.track), _p(self.begin), _p(self.len), _p(self.cap)]

    def run_of(self, begin):
        return int(np.searchsorted(self.begin, begin, side="right") - 1)


def cost_balanced(lib, runs, target, c0):
    n = int(runs.len.sum())
    out, slow = np.zeros((n, 3), np.int64), np.zeros(1, np.float32)
    k = lib.sch_cost_balanced(*runs.args(), _p(runs.w), target, c0, _p(out), n, _p(slow))
    return out[:k], float(slow[0])


def reweigh(lib, runs, tiles, ns, weighted, target):
    n = int(runs.len.sum())
    out, bal, wt = np.zeros((n, 3), np.int64), np.zeros(2, np.float32), np.array([int(weighted)], np.int32)
    tiles = np.ascontiguousarray(tiles, np.int64)
    ns = np.ascontiguousarray(ns, np.uint32)
    k = lib.sch_reweigh(*runs.args(), _p(runs.w), len(tiles), _p(tiles), _p(ns), _p(wt), target, _p(out), n, _p(bal))
    return (None if k < 0 else out[:k]), bool(wt[0]), tuple(float(b) for b in bal)


def track_ids(lens, order=None):
    order = range(len(lens)) if order is None else order
    return np.concatenate([np.full(l, t, np.int32) for t, l in zip(order, lens)])


def check_partition(tiles, tid, cap):
    """the tiles cover [0, n) exactly once, each within one track's run, 1 <= count <= cap"""
    assert len(tiles) > 0
    srt = tiles[np.argsort(tiles[:, 2], kind="stable")]
    assert srt[0, 2] == 0 and srt[-1, 2] + srt[-1, 1] == len(tid)
    assert np.array_equal(srt[1:, 2], srt[:-1, 2] + srt[:-1, 1]), "gaps or overlaps"
    assert (tiles[:, 1] >= 1).all() and (tiles[:, 1] <= cap).all()
    for track, count, begin in tiles:
        assert (tid[begin:begin + count] == track).all(), "a tile spans two tracks"


BENCH_LENS = [2849] * 22 + [65536 - 22 * 2849]  # the benchmark's population: 65,536 agents over 23 tracks
SHAPES = [
    pytest.param(BENCH_LENS, 512, 148, id="bench"),
    pytest.param([1], 256, 148, id="one-agent"),
    pytest.param([5, 3, 1, 7], 64, 148, id="more-ctas-than-agents"),
    pytest.param([40, 7, 90, 3, 300], 16, 4, id="runs-shorter-than-a-tile"),
    pytest.param([1000, 999, 1001], 37, 8, id="several-waves"),
]


@pytest.mark.parametrize("lens,big,ctas", SHAPES)
@pytest.mark.parametrize("tail_div", [0, 1, 4])
def test_guided_tiles_partition_in_order(lib, lens, big, ctas, tail_div):
    tid = track_ids(lens, order=[(3 * i) % 23 for i in range(len(lens))])
    tiles = guided(lib, tid, big, ctas, tail_div)
    check_partition(tiles, tid, big)
    n = len(tid)
    if tail_div > 1:  # the small tiles follow the big ones and hold every run's share of the tail
        small = max(1, big // tail_div)
        tail = sum(l * min(n // 2, ctas * big // 2) // n for l in lens)
        k = len(tiles)
        while k > 0 and tiles[k - 1, 1] <= small:
            k -= 1
        assert tiles[k:, 1].sum() >= tail
    else:  # uniform: in agent order, every run cut into tiles of `big`, only its last one shorter
        assert (np.diff(tiles[:, 2]) > 0).all()
        assert len(tiles) == sum(-(-l // big) for l in lens)


@pytest.mark.parametrize("lens,big,ctas", SHAPES)
@pytest.mark.parametrize("waves", [1, 3])
def test_balanced_tiles_partition_and_target(lib, lens, big, ctas, waves):
    tid = track_ids(lens)
    tiles, target = balanced(lib, tid, big, ctas, waves)
    check_partition(tiles, tid, big)
    n = len(tid)
    assert target % ctas == 0 and target >= waves * ctas
    assert target >= -(-n // big) and target >= sum(-(-l // big) for l in lens)
    assert len(tiles) == min(target, n)  # every run gets tiles until the target is reached or every tile is one agent
    # a run is cut into equal parts
    for t in range(len(lens)):
        counts = tiles[tiles[:, 0] == t, 1]
        assert counts.max() - counts.min() <= 1
    # largest first
    assert (np.diff(tiles[:, 1]) <= 0).all()
    if lens is BENCH_LENS and waves == 1:
        assert target == ctas and len(tiles) == ctas


def plain_balanced(lens, cap, target):
    """reference: the balanced tiling by agent count, one more tile at a time for the run with the largest tiles"""
    k = [max(1, -(-l // cap)) for l in lens]
    while sum(k) < target:
        best = None
        for r, l in enumerate(lens):
            if l > k[r] and (best is None or -(-l // k[r]) > -(-lens[best] // k[best])):
                best = r
        if best is None:
            break
        k[best] += 1
    begin = np.concatenate([[0], np.cumsum(lens)[:-1]])
    tiles = [(r, (l * (t + 1)) // k[r] - (l * t) // k[r], begin[r] + (l * t) // k[r]) for r, l in enumerate(lens) for t in range(k[r])]
    tiles = [t for t in tiles if t[1] > 0]
    return np.array(sorted(tiles, key=lambda t: -t[1]), np.int64)  # sorted() is stable


@pytest.mark.parametrize("lens,cap,target", [([7, 3, 12, 5], 4, 10), (BENCH_LENS, 512, 148), ([100], 7, 3), ([2, 2, 2], 8, 20)])
def test_cost_balanced_with_unit_weights_is_the_plain_balanced_tiling(lib, lens, cap, target):
    runs = Runs(lens, cap)
    tiles, slow = cost_balanced(lib, runs, target, 0.0)
    assert np.array_equal(tiles, plain_balanced(lens, cap, target))
    assert slow >= 1.0


def tile_costs(runs, tiles, c0):
    return np.array([c0 + runs.w[runs.run_of(b)] * c for _, c, b in tiles])


@pytest.mark.parametrize("seed", range(12))
def test_cost_balanced_minimises_the_slowest_tile(lib, seed):
    rng = np.random.default_rng(seed)
    lens = rng.integers(1, 9, size=int(rng.integers(1, 4))).tolist()
    cap = int(rng.integers(1, 6))
    runs = Runs(lens, cap, w=rng.uniform(0.5, 2.0, len(lens)))
    c0 = float(rng.uniform(0, 5))
    target = int(rng.integers(1, sum(lens) + 3))
    tiles, slow = cost_balanced(lib, runs, target, c0)
    check_partition(tiles, track_ids(lens), cap)
    costs = tile_costs(runs, tiles, c0)
    assert (np.diff(costs) <= 1e-9).all(), "most expensive first"
    assert slow >= 1.0 and slow == pytest.approx(costs.max() * len(costs) / costs.sum(), rel=1e-6)
    # brute force over every split: a run of `l` agents in `k` parts has a part of at least ceil(l / k) agents, and no part may
    # exceed the cap; at most max(target, tiles the caps force) parts in all
    lo = [-(-l // cap) for l in lens]
    budget = max(target, sum(lo))
    best = min(max(c0 + runs.w[r] * -(-l // k[r]) for r, l in enumerate(lens))
               for k in itertools.product(*[range(a, l + 1) for a, l in zip(lo, lens)]) if sum(k) <= budget)
    assert costs.max() == pytest.approx(best, rel=1e-12)


def _measured(runs, tiles, ray_per_agent, rest):
    """tile times as the kernel reports them: ray phase = w_true(run) * count, the rest given per tile"""
    ns = np.zeros((len(tiles), 2), np.uint32)
    for i, (_, c, b) in enumerate(tiles):
        ns[i] = (ray_per_agent[runs.run_of(b)] * c, rest[i])
    return ns


def test_reweigh_first_round_takes_the_measured_weights_and_c0_is_the_median(lib):
    runs = Runs([600, 300, 900], 256)
    target = 12
    tiles, _ = cost_balanced(lib, runs, target, 0.0)
    true_w = np.array([10.0, 30.0, 20.0])
    rest = np.arange(len(tiles)) * 100 + 1000  # median of these is c0
    ns = _measured(runs, tiles, true_w, rest)
    new, weighted, (before, after) = reweigh(lib, runs, tiles, ns, False, target)
    assert weighted and new is not None
    assert np.allclose(runs.w, true_w)
    c0 = float(np.sort(rest)[len(rest) // 2])
    tot = ns.astype(np.float64).sum(1)
    assert before == pytest.approx(tot.max() * len(tot) / tot.sum(), rel=1e-6)
    want, want_after = cost_balanced(lib, Runs([600, 300, 900], 256, w=true_w), target, c0)
    assert np.array_equal(new, want) and after == pytest.approx(want_after, rel=1e-6)
    _, other_after = cost_balanced(lib, Runs([600, 300, 900], 256, w=true_w), target, c0 + 500)
    assert other_after != pytest.approx(after, rel=1e-6), "the case does not tell c0 apart"


def test_reweigh_later_rounds_go_half_way(lib):
    runs = Runs([500, 500], 128, w=[4.0, 8.0])
    target = 8
    tiles, _ = cost_balanced(lib, runs, target, 0.0)
    ns = _measured(runs, tiles, np.array([12.0, 2.0]), np.full(len(tiles), 700))
    new, weighted, _ = reweigh(lib, runs, tiles, ns, True, target)
    assert weighted and new is not None
    assert np.allclose(runs.w, [0.5 * (4 + 12), 0.5 * (8 + 2)])


def test_reweigh_ignores_unmeasured_and_wrapped_tiles(lib):
    runs = Runs([400, 400, 400], 100)
    target = 12
    tiles, _ = cost_balanced(lib, runs, target, 0.0)
    assert len(tiles) == 12
    true_w = np.array([5.0, 6.0, 7.0])
    rest = np.full(len(tiles), 300)
    ns = _measured(runs, tiles, true_w, rest)
    # one tile of run 0 never ran, one of run 1 has a wrapped timer: neither may move the weights or c0
    r0 = [i for i, t in enumerate(tiles) if runs.run_of(t[2]) == 0][0]
    r1 = [i for i, t in enumerate(tiles) if runs.run_of(t[2]) == 1][0]
    ns[r0] = (0, 4_000_000_000)
    ns[r1] = (2_000_000_000, 4_000_000_000)
    new, _, (_, after) = reweigh(lib, runs, tiles, ns, False, target)
    assert new is not None and np.allclose(runs.w, true_w)
    _, want_after = cost_balanced(lib, Runs([400, 400, 400], 100, w=true_w), target, 300.0)
    assert after == pytest.approx(want_after, rel=1e-6)


def test_reweigh_needs_half_the_tiles_measured(lib):
    runs = Runs([300, 300], 64, w=[3.0, 4.0])
    target = 10
    tiles, _ = cost_balanced(lib, runs, target, 0.0)
    ns = _measured(runs, tiles, np.array([9.0, 9.0]), np.full(len(tiles), 100))
    ns[: len(tiles) // 2 + 1, 0] = 0  # fewer than half measured
    new, weighted, _ = reweigh(lib, runs, tiles, ns, False, target)
    assert new is None and not weighted and np.allclose(runs.w, [3.0, 4.0])
    ns[len(tiles) // 2, 0] = 9 * tiles[len(tiles) // 2, 1]  # exactly half
    new, weighted, _ = reweigh(lib, runs, tiles, ns, False, target)
    assert new is not None and weighted

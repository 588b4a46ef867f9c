"""CPU: the sizing of a population and the tilings of the agent range (openkitchen_b200/csrc/ok_schedule.cpp), compiled
with g++ next to a small C wrapper and driven through ctypes.  Guided and balanced tilings must partition the agents into
same-track tiles within their caps; the cost-balanced tiling must minimise the slowest tile; the feedback model must
ignore what carries no information and damp what it learns.  The sizing must choose the kernel shape and the tilings the
library chose on a B200 (tests/golden/sizing_plans.json, tools/make_golden_sizing.py) and keep its rules."""
import ctypes as C
import itertools
import json
import os
import subprocess

import numpy as np
import pytest

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "openkitchen_b200", "csrc")

WRAPPER = r'''
#include "ok_schedule.hpp"
#include <climits>
#include <cstdio>
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
// k[10]: the knobs in SizingKnobs order, INT_MIN = unset; k[1] (OK_BEAM_KERNEL): 0 automatic, 1 staged, 2 unstaged
ok::SizingKnobs knobs_of(const int *k)
{
    auto opt = [](int v) { return v == INT_MIN ? std::optional<int>() : std::optional<int>(v); };
    ok::SizingKnobs s;
    s.batch_agents      = opt(k[0]);
    s.beam_kernel       = static_cast<ok::SizingKnobs::BeamKernel>(k[1] == INT_MIN ? 0 : k[1]);
    s.beam_batch_agents = opt(k[2]);
    s.beam_tail         = opt(k[3]);
    s.beam_waves        = opt(k[4]);
    s.auto_balance      = opt(k[5]);
    s.e2e_tiles         = opt(k[6]);
    s.e2e_tiles_q16     = opt(k[7]);
    s.e2e_flushers      = opt(k[8]);
    s.act_stage         = opt(k[9]);
    return s;
}
ok::StepFootprint footprint_of(const int64_t *f)
{
    return {f[0], f[1], f[2], static_cast<int32_t>(f[3]), static_cast<int32_t>(f[4]), static_cast<int32_t>(f[5])};
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

// dev: num_sms, smem_optin, max_blob.  shape[8]: batch_agents, smem, beam_staged, beam_block, batch_agents_beam, smem_beam,
// auto_balance, act_stage.  Returns 0, or -1 with the error in err.
int sch_size(int64_t n, int rays, const int64_t *dev, const int64_t *fp, const int *knobs, int64_t *shape, char *err, int err_cap)
{
    ok::Sizing  s;
    std::string why;
    if (!ok::size_population(n, rays, static_cast<int>(dev[0]), static_cast<int>(dev[1]), static_cast<size_t>(dev[2]), footprint_of(fp),
                             knobs_of(knobs), s, why))
    {
        std::snprintf(err, err_cap, "%s", why.c_str());
        return -1;
    }
    const int64_t v[8] = {s.batch_agents, static_cast<int64_t>(s.smem), s.beam_staged, s.beam_block, s.batch_agents_beam,
                          static_cast<int64_t>(s.smem_beam), s.auto_balance, s.act_stage};
    std::memcpy(shape, v, sizeof v);
    return 0;
}

// tiling `which` (0 grid, 1 beam, 2 e2e, 3 q16) of the population sized as sch_size does, with `ctas_per_sm` unstaged beam
// CTAs per SM.  info[5]: the tiling's ctas and capacity, feedback, target, e2e_flushers.
int64_t sch_tiling(const int32_t *track_id, int64_t n, int rays, const int64_t *dev, const int64_t *fp, const int *knobs, int ctas_per_sm,
                   int which, int64_t *out, int64_t cap, int64_t *info)
{
    ok::Sizing  s;
    std::string why;
    if (!ok::size_population(n, rays, static_cast<int>(dev[0]), static_cast<int>(dev[1]), static_cast<size_t>(dev[2]), footprint_of(fp),
                             knobs_of(knobs), s, why))
        return -1;
    s.ctas_per_sm_beam          = s.beam_staged ? 1 : ctas_per_sm;
    const ok::PopulationTilings t = ok::tile_population(track_id, n, s, static_cast<int>(dev[0]), knobs_of(knobs));
    const ok::Tiling           &r = which == 0 ? t.grid : which == 1 ? t.beam : which == 2 ? t.e2e : t.q16;
    const int64_t               v[5] = {r.ctas, static_cast<int64_t>(r.capacity), t.feedback, t.target, t.e2e_flushers};
    std::memcpy(info, v, sizeof v);
    return put(r.tiles, out, cap);
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
    L.sch_size.restype, L.sch_tiling.restype = C.c_int, C.c_int64
    L.sch_size.argtypes = [C.c_int64, C.c_int, _P, _P, _P, _P, C.c_char_p, C.c_int]
    L.sch_tiling.argtypes = [_P, C.c_int64, C.c_int, _P, _P, _P, C.c_int, C.c_int, _P, C.c_int64, _P]
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


# ---- sizing of a population -----------------------------------------------------------------------------------------

# the step kernels' footprint (ok_step.cuh, ok_device.cuh): sizeof(AgentRec), batch_smem_bytes' bytes per ray,
# beam_static_smem(true), beam_block(true), beam_block(false), OK_BEAM_TILE
FOOTPRINT = np.array([64, 8, 42112, 1024, 256, 64], np.int64)
# occupancy of the unstaged beam kernel (256 threads, 64 registers): the plan "bench-unstaged" runs 592 = 148 x 4 CTAs
UNSTAGED_CTAS_PER_SM = 4
KNOBS = ["OK_BATCH_AGENTS", "OK_BEAM_KERNEL", "OK_BEAM_BATCH_AGENTS", "OK_BEAM_TAIL", "OK_BEAM_WAVES", "OK_AUTO_BALANCE",
         "OK_E2E_TILES", "OK_E2E_TILES_Q16", "OK_E2E_FLUSHERS", "OK_ACT_STAGE"]
UNSET = -(2 ** 31)
SHAPE = ["batch_agents", "smem", "beam_staged", "beam_block", "batch_agents_beam", "smem_beam", "auto_balance", "act_stage"]
with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "sizing_plans.json")) as _f:
    GOLDEN = json.load(_f)
B200 = GOLDEN["device"]


def knob_array(knobs):
    """the variables as ok_capi.cu reads them (atoi; OK_BEAM_KERNEL by name)"""
    def value(k, v):
        if k == "OK_BEAM_KERNEL":
            return {"staged": 1, "unstaged": 2}.get(v, 0)
        return int(v)
    return np.array([value(k, knobs[k]) if k in knobs else UNSET for k in KNOBS], np.int32)


def device(num_sms=None, smem_optin=None, max_blob=None):
    return np.array([num_sms or B200["num_sms"], smem_optin or B200["smem_optin"], max_blob or B200["max_blob"]], np.int64)


def size(lib, n, rays, knobs=None, **dev):
    shape, err = np.zeros(len(SHAPE), np.int64), C.create_string_buffer(256)
    if lib.sch_size(n, rays, _p(device(**dev)), _p(FOOTPRINT), _p(knob_array(knobs or {})), _p(shape), err, 256) != 0:
        return err.value.decode()
    return dict(zip(SHAPE, shape.tolist()))


TILINGS = {"grid": 0, "beam": 1, "e2e": 2, "q16": 3}


def tiling(lib, tid, rays, which, knobs=None, ctas_per_sm=UNSTAGED_CTAS_PER_SM, **dev):
    out, info = np.zeros((len(tid), 3), np.int64), np.zeros(5, np.int64)
    k = lib.sch_tiling(_p(tid), len(tid), rays, _p(device(**dev)), _p(FOOTPRINT), _p(knob_array(knobs or {})), ctas_per_sm,
                       TILINGS[which], _p(out), len(tid), _p(info))
    assert k >= 0
    return out[:k], dict(zip(["ctas", "capacity", "feedback", "target", "flushers"], info.tolist()))


def golden_tid(n):
    return (np.arange(n) * 23 // n).astype(np.int32)  # tools/make_golden_sizing.py: 23 tracks, contiguous


@pytest.mark.parametrize("name", list(GOLDEN["plans"]))
def test_plan_is_the_one_chosen_on_b200(lib, name):
    """launch_stats() and debug_tiles() of the library right after alloc_agents, minted on a B200"""
    p = GOLDEN["plans"][name]
    shape = size(lib, p["n"], p["rays"], p["knobs"])
    which = "beam" if p["raycast"] == "beam" else "grid"
    tiles, info = tiling(lib, golden_tid(p["n"]), p["rays"], which, p["knobs"])
    grid = max(1, min(info["ctas"], len(tiles)))  # ok_capi.cu: schedule_grid
    if which == "beam":
        assert (grid, shape["beam_block"], shape["smem_beam"], len(tiles)) == (p["grid"], p["block"], p["smem"], p["tiles"])
        assert np.array_equal(tiles, np.asarray(p["debug_tiles"], np.int64).reshape(-1, 3))
    else:
        assert (grid, 1024, shape["smem"], len(tiles)) == (p["grid"], p["block"], p["smem"], p["tiles"])


E2E_SHAPES = [
    pytest.param(65536, 32, {}, id="bench"),
    pytest.param(65536, 32, {"OK_E2E_FLUSHERS": "8"}, id="flushers8"),
    pytest.param(65536, 32, {"OK_E2E_FLUSHERS": "500"}, id="flushers-capped"),
    pytest.param(300, 32, {"OK_BEAM_KERNEL": "staged", "OK_E2E_TILES": "6"}, id="300-staged"),
    pytest.param(8192, 5, {"OK_BEAM_BATCH_AGENTS": "40", "OK_E2E_TILES_Q16": "2"}, id="8192x5"),
]


@pytest.mark.parametrize("n,rays,knobs", E2E_SHAPES)
def test_e2e_tilings_partition_the_agents_over_their_ctas(lib, n, rays, knobs):
    tid = golden_tid(n)
    shape = size(lib, n, rays, knobs)
    assert shape["beam_staged"] == 1
    flushers = min(int(knobs.get("OK_E2E_FLUSHERS", 0)), B200["num_sms"] // 2)
    for which, ctas in [("e2e", B200["num_sms"] - flushers), ("q16", B200["num_sms"])]:
        tiles, info = tiling(lib, tid, rays, which, knobs)
        check_partition(tiles, tid, shape["batch_agents_beam"])
        assert info["flushers"] == flushers and info["ctas"] == ctas
        assert info["capacity"] % ctas == 0 and len(tiles) <= info["capacity"]  # capacity: the balanced tiling's target


@pytest.mark.parametrize("knobs,e2e,q16", [({}, 4, 3), ({"OK_E2E_TILES": "6"}, 6, 6), ({"OK_E2E_TILES_Q16": "2"}, 4, 2),
                                           ({"OK_E2E_TILES": "6", "OK_E2E_TILES_Q16": "2"}, 6, 2), ({"OK_E2E_TILES": "0"}, 1, 1)])
def test_q16_tiles_follow_e2e_tiles_only_when_unset(lib, knobs, e2e, q16):
    tid = golden_tid(65536)  # the bench population: one tile per CTA and wave
    for which, per_cta in [("e2e", e2e), ("q16", q16)]:
        tiles, info = tiling(lib, tid, 32, which, knobs)
        assert info["capacity"] == per_cta * B200["num_sms"] and len(tiles) == info["capacity"]


def test_unstaged_population_has_no_e2e_tiling_and_a_guided_beam_tiling(lib):
    tid = golden_tid(300)
    assert size(lib, 300, 32)["beam_staged"] == 0
    assert len(tiling(lib, tid, 32, "e2e")[0]) == 0 and len(tiling(lib, tid, 32, "q16")[0]) == 0
    tiles, info = tiling(lib, tid, 32, "beam")
    assert not info["feedback"] and info["ctas"] == B200["num_sms"] * UNSTAGED_CTAS_PER_SM and info["capacity"] == 0


def test_knob_flags_and_caps(lib):
    bench = size(lib, 65536, 32)
    assert bench["auto_balance"] == 1 and bench["act_stage"] == 1
    off = size(lib, 65536, 32, {"OK_AUTO_BALANCE": "0", "OK_ACT_STAGE": "0"})
    assert off["auto_balance"] == 0 and off["act_stage"] == 0
    # OK_BATCH_AGENTS limits only the grid kernel's batch
    capped = size(lib, 65536, 32, {"OK_BATCH_AGENTS": "7"})
    assert capped["batch_agents"] == 7 and capped["batch_agents_beam"] == bench["batch_agents_beam"]
    # tile-local ray indices are 16 bits: at most 65535 / rays agents per beam tile
    assert size(lib, 65536, 1024, {"OK_BEAM_KERNEL": "staged"})["batch_agents_beam"] == 65535 // 1024


@pytest.mark.parametrize("kernel", ["staged", "unstaged"])
def test_too_little_shared_memory_is_a_capacity_error(lib, kernel):
    """in both shapes, the beam kernel's static shared memory and 4 KB must fit next to the largest track (rounded up to
    128 bytes) and its own 4 KB"""
    blob = 146784
    need = (blob + 127) // 128 * 128 + 4096 + int(FOOTPRINT[2]) + 4096
    err = size(lib, 300, 32, {"OK_BEAM_KERNEL": kernel}, smem_optin=need - 1, max_blob=blob)
    assert err == "shared memory cannot hold one agent's rays next to the largest track"
    assert size(lib, 300, 32, {"OK_BEAM_KERNEL": kernel}, smem_optin=need, max_blob=blob)["batch_agents"] >= 1

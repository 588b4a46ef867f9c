"""GPU: size-independent properties at BASELINE's full size (65,536 agents x 32 rays x 23 tracks), where the
CPU oracle is too slow to shadow every agent: beam lists == grid == brute force on every ray, obs/hit consistency, a
sampled slice against the oracle, determinism."""
import numpy as np
import pytest

import bench
import openkitchen_b200 as ok
from oracle.api import Oracle

pytestmark = pytest.mark.gpu
N = 65536


def _run(raycast, ticks):
    env = ok.Env(device=0, movement_mode=ok.MOVE_VELOCITY, reward_mode=ok.REWARD_CMAES_PROGRESS, auto_reset=1,
                 raycast_mode=raycast)
    bench.build_workload(ok, env, N)
    env.launch_steps_random(0, ticks)
    env.sync()
    return env


def test_full_size_grid_equals_brute_force_and_is_deterministic():
    ticks = 25
    a = _run(ok.RAYCAST_BEAM, ticks)
    b = _run(ok.RAYCAST_BRUTE, ticks)
    c = _run(ok.RAYCAST_BEAM, ticks)
    d = _run(ok.RAYCAST_GRID, ticks)
    for name in ok.BUFFERS:
        x, y, z, w = a.read(name), b.read(name), c.read(name), d.read(name)
        assert np.array_equal(x.view(np.uint8), y.view(np.uint8)), f"beam lists vs brute force: {name}"
        assert np.array_equal(w.view(np.uint8), y.view(np.uint8)), f"grid vs brute force: {name}"
        assert np.array_equal(x.view(np.uint8), z.view(np.uint8)), f"run-to-run: {name}"
    # invariants of the outputs
    obs, t, seg, rel = a.read("obs"), a.read("hit_t"), a.read("hit_seg"), a.read("hit_rel")
    assert ((t >= 0) & (t <= 200.0)).all() and ((seg >= -1)).all()
    assert ((seg == -1) == (t == 200.0)).mean() > 0.999  # a miss reports the sensor range
    assert np.allclose(obs * 200.0, np.sqrt((rel.astype(np.float64) ** 2).sum(-1)), rtol=1e-5, atol=1e-4)
    crashed = a.read("crashed").astype(bool)
    assert (a.read("min_dist2")[crashed & ~a.read("timed_out").astype(bool)] < 2.0).all()
    assert 0 < crashed.mean() < 0.2


def test_full_size_sampled_slice_matches_oracle():
    """agents are independent, so a slice of the big batch must evolve exactly like the same agents alone"""
    ticks = 40
    env = _run(ok.RAYCAST_BEAM, ticks)
    names = ok.track_names()
    sel = np.arange(0, N, 997)[:64]
    tid_all = (np.arange(N, dtype=np.int64) * 23 // N).astype(np.int32)
    ora = Oracle("port", movement_mode=0, reward_mode=2, auto_reset=1)
    pts_per = []
    for nm in names:
        cols = ok.track_columns(nm)
        ora.add_track(cols)
        pts_per.append(len(cols[0]))
    # the oracle's Philox counter is the agent index, so give it the same ids by placing the sampled agents
    # at their global positions in a sparse population: simulate only `sel`, feeding the product's own actions
    ora.alloc_agents(len(sel), ok.ray_fan(32), tid_all[sel])
    ids = sel.astype(np.uint64)
    pts = ((ids * np.uint64(2654435761)) % np.uint64(2**32) % np.asarray(pts_per, dtype=np.uint64)[tid_all[sel]]).astype(np.int32)
    ora.reset(None, pts)
    env2 = ok.Env(device=0, movement_mode=0, reward_mode=2, auto_reset=1)
    bench.build_workload(ok, env2, N)
    for s in range(ticks):
        env2.fill_random_actions(s)
        thr, st = env2.read("act_throttle")[sel], env2.read("act_steer")[sel]
        env2.launch_step()
        ora.step(thr, st)
    for name in ("pos_x", "pos_y", "rot", "crashed", "hit_seg", "hit_t", "obs", "reward", "fitness", "nearest_idx"):
        got, want = env2.read(name)[sel], ora.buffer(name)
        assert np.array_equal(got.view(np.uint8), want.view(np.uint8)), name
        assert np.array_equal(env.read(name)[sel].view(np.uint8), want.view(np.uint8)), name + " (fused random actions)"


def test_tile_schedules_give_the_same_bits(monkeypatch):
    """the results do not depend on how the agents are cut into tiles: the default balanced tiling (about one large tile
    per CTA), small 96-agent tiles (phase 4 then runs four lanes per agent instead of one thread) and the guided
    schedule with a tail of quarter-size tiles must agree bit for bit"""
    ticks = 20
    a = _run(ok.RAYCAST_BEAM, ticks)
    monkeypatch.setenv("OK_BEAM_BATCH_AGENTS", "96")
    b = _run(ok.RAYCAST_BEAM, ticks)
    monkeypatch.setenv("OK_BEAM_BATCH_AGENTS", "256")
    monkeypatch.setenv("OK_BEAM_TAIL", "4")
    c = _run(ok.RAYCAST_BEAM, ticks)
    assert b.launch_stats().tiles > a.launch_stats().tiles and c.launch_stats().tiles > a.launch_stats().tiles
    for name in ok.BUFFERS:
        assert np.array_equal(a.read(name).view(np.uint8), b.read(name).view(np.uint8)), f"96-agent tiles: {name}"
        assert np.array_equal(a.read(name).view(np.uint8), c.read(name).view(np.uint8)), f"quarter-size tail: {name}"


@pytest.mark.parametrize("kernel", ["staged"])
def test_feedback_tiling_changes_the_schedule_not_the_bits(monkeypatch, kernel):
    """ok_balance_schedule re-cuts the tiles from the tile times the kernel measured (the library also does it on its own
    after the 16th and 64th launch): the tiling changes, tiles stay within their tracks and cover every agent once, and
    the results are those of a run that never re-balanced, bit for bit"""
    monkeypatch.setenv("OK_BEAM_KERNEL", kernel)
    ticks = 80
    monkeypatch.setenv("OK_AUTO_BALANCE", "0")
    a = _run(ok.RAYCAST_BEAM, ticks)
    monkeypatch.setenv("OK_AUTO_BALANCE", "1")
    b = _run(ok.RAYCAST_BEAM, ticks)  # re-balanced by the library at launches 16 and 64
    monkeypatch.setenv("OK_AUTO_BALANCE", "0")
    c = ok.Env(device=0, movement_mode=ok.MOVE_VELOCITY, reward_mode=ok.REWARD_CMAES_PROGRESS, auto_reset=1)
    tid = bench.build_workload(ok, c, N)
    before = c.debug_tiles().copy()
    for t in range(ticks):
        c.launch_steps_random(t, 1)
        if t in (5, 30, 31):
            worst_before, worst_after = c.balance_schedule()
            assert worst_before >= 1.0 and 1.0 <= worst_after < worst_before + 0.05
    c.sync()
    for env in (b, c):
        tiles = env.debug_tiles()
        assert not np.array_equal(tiles, a.debug_tiles()), "the tiling never changed"
        order = np.argsort(tiles[:, 2])
        tr, cnt, beg = tiles[order].T
        assert beg[0] == 0 and (beg[1:] == beg[:-1] + cnt[:-1]).all() and beg[-1] + cnt[-1] == N, "tiles do not partition the agents"
        assert all((tid[b0:b0 + n] == t).all() for t, n, b0 in tiles), "a tile spans two tracks"
        assert cnt.max() <= env.launch_stats().block_threads
        for name in ok.BUFFERS:
            assert np.array_equal(a.read(name).view(np.uint8), env.read(name).view(np.uint8)), name
    assert len(before) == len(a.debug_tiles())


def test_feedback_tiling_under_a_captured_graph(monkeypatch):
    """a CUDA graph captured BEFORE a re-balancing keeps replaying correctly after it: the graph reads the tile table and
    the first-tile records at every replay, the re-balancing rewrites both together.  Several tiles per CTA
    (OK_BEAM_WAVES=3), where a CTA mixes its first-tile record with later tiles from the table."""
    import torch

    monkeypatch.setenv("OK_BEAM_WAVES", "3")
    monkeypatch.setenv("OK_AUTO_BALANCE", "0")
    ticks_per_replay, replays = 4, 6

    def make():
        env = ok.Env(device=0, movement_mode=ok.MOVE_VELOCITY, reward_mode=ok.REWARD_CMAES_PROGRESS, auto_reset=1)
        bench.build_workload(ok, env, N)
        return env

    ref = make()
    ref.launch_steps_random(0, 2)  # (the graphed env's two warm-up ticks)
    env = make()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        env.launch_steps_random(0, 2, bench.SEED, side.cuda_stream)
    side.synchronize()
    assert env.launch_stats().tiles > 2 * env.launch_stats().grid_blocks
    graph = torch.cuda.CUDAGraph()
    # the graph replays the SAME tick numbers every time (the step counter is baked in): compare with a reference that does too
    with torch.cuda.graph(graph, stream=side):
        env.launch_steps_random(1000, ticks_per_replay, bench.SEED, side.cuda_stream)
    before = env.debug_tiles().copy()
    for r in range(replays):
        graph.replay()
        torch.cuda.synchronize()
        if r in (1, 3):
            env.balance_schedule()
        ref.launch_steps_random(1000, ticks_per_replay)
    ref.sync()
    torch.cuda.synchronize()
    assert not np.array_equal(before, env.debug_tiles()), "the tiling never changed"
    for name in ok.BUFFERS:
        assert np.array_equal(env.read(name).view(np.uint8), ref.read(name).view(np.uint8)), name


@pytest.mark.parametrize("raycast,n", [(ok.RAYCAST_BEAM, 300), (ok.RAYCAST_GRID, 4096), (ok.RAYCAST_BEAM, 4096)])
def test_balance_schedule_is_harmless_everywhere(raycast, n):
    """ok_balance_schedule before any launch, on the unstaged shape (no feedback there), in grid mode, and repeatedly on a
    staged population with a single track: never an error, never a changed result"""
    names = ["Monza"] if n == 4096 and raycast == ok.RAYCAST_BEAM else ["Monza", "Spa", "Sochi"]
    tid = (np.arange(n) * len(names) // n).astype(np.int32)

    def make():
        env = ok.Env(device=0, reward_mode=ok.REWARD_CMAES_PROGRESS, auto_reset=1, raycast_mode=raycast)
        for nm in names:
            env.add_named_track(nm)
        env.alloc_agents(n, ok.ray_fan(32), tid)
        return env

    a, b = make(), make()
    b.balance_schedule()  # nothing measured yet
    for t in range(40):
        a.launch_steps_random(t, 1)
        b.launch_steps_random(t, 1)
        if t % 7 == 3:
            before, after = b.balance_schedule()
            assert before >= 0.0 and after >= 0.0
    a.sync()
    b.sync()
    for name in ok.BUFFERS:
        assert np.array_equal(a.read(name).view(np.uint8), b.read(name).view(np.uint8)), name

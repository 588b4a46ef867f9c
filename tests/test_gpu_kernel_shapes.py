"""GPU: the beam kernel and the lidar query at the shapes the other parity files never reach.  Pass A's ray queue filled
past its capacity in both kernel shapes; phase 4 with one thread per agent (tiles of more than 512 agents) in the plain,
drawn and laps variants, forced and as the balanced tiling cuts a large population; the staged kernel, the grid and the
brute-force kernel at ray counts from 1 to 1,024; and ok_lidar_query in each of its three thread mappings.  Every
comparison is bit for bit against the port oracle (or the agent path, for the query) on every buffer, and every test
first asserts, from the library's own counters and tilings, that it runs the shape it is named for."""
import numpy as np
import pytest

import bench
import openkitchen_b200 as ok
from oracle.api import Oracle
from tests.laps_oracle import Laps
from tests.reset_draws_oracle import DrawnResets
from tests.test_gpu_laps import assert_laps, plant
from tests.test_gpu_lidar_query import C_NAMES, MODES, NAMES, _hard_poses
from tests.test_gpu_parity_gaps import _oracle_slice
from tests.util import ALL_BUFS, assert_same, make_pair, same_bits, spread_points

pytestmark = pytest.mark.gpu

SEED = 0x5A9E
# rays pass A can queue for pass B per CTA, staged / unstaged kernel (beam_pend_cap, openkitchen_b200/csrc/ok_step.cuh:291-294);
# an append past it finishes the ray on the spot (process_full in pass A)
PEND_CAP = {"staged": 8192, "unstaged": 2048}
BLOCK = {"staged": 1024, "unstaged": 256}


def no_violations(env):
    n, _ = env.debug_violations()
    assert n == 0, f"{n} out-of-range indices counted"


def force(monkeypatch, **knobs):
    """the sizing knobs of ok_alloc_agents (read at every alloc) for this test"""
    for k, v in knobs.items():
        monkeypatch.setenv(k, str(v))


def step_pair(env, ora, step):
    env.launch_steps_random(step, 1)
    ora.fill_random_actions(step)
    ora.step()


def guided_counts(tid, batch):
    """tile sizes of the guided tiling without a tail (OK_BEAM_TAIL=0): each track run cut into tiles of `batch` agents,
    the last one shorter"""
    out = []
    for t in dict.fromkeys(tid.tolist()):
        run = int((tid == t).sum())
        out += [batch] * (run // batch) + ([run % batch] if run % batch else [])
    return out


# ---------------------------------------------------------------------------------------------------------------------
# A. pass A's queue overflows
# ---------------------------------------------------------------------------------------------------------------------
def off_lane_poses(env, tid, rng):
    """Per agent a pose 8-40 px beyond one side of its track's lane, farther than (lane half-width + 4 px + 4 px) from every
    centre-line point: the beam table covers the cells within half-width + 4 px of a centre-line point (beam_plan,
    ok_beam.cpp), so the lidar origin's 2 px cell is not covered and every ray of the agent is queued by pass A, while the
    lane's wall is a few tens of pixels away."""
    n = len(tid)
    x, y = np.empty(n, np.float32), np.empty(n, np.float32)
    for t in np.unique(tid):
        cx, cy = env.track_array(int(t), "x").astype(np.float64), env.track_array(int(t), "y").astype(np.float64)
        r = np.maximum(env.track_array(int(t), "w_left"), env.track_array(int(t), "w_right")).astype(np.float64) + 4.0
        tx, ty = np.roll(cx, -1) - np.roll(cx, 1), np.roll(cy, -1) - np.roll(cy, 1)
        ln = np.hypot(tx, ty)
        nx, ny = -ty / ln, tx / ln
        agents = np.flatnonzero(tid == t)
        m = 4 * len(agents)
        i = rng.integers(0, len(cx), m)
        side = rng.choice([-1.0, 1.0], m)
        d = r[i] + rng.uniform(8.0, 40.0, m)
        px, py = cx[i] + side * nx[i] * d, cy[i] + side * ny[i] * d
        clear = (np.hypot(px[:, None] - cx[None, :], py[:, None] - cy[None, :]) - r[None, :]).min(axis=1) > 4.0
        keep = np.flatnonzero(clear)[:len(agents)]
        assert len(keep) == len(agents), "too few off-lane poses"
        x[agents], y[agents] = px[keep], py[keep]
    rot = rng.uniform(-180.0, 180.0, n).astype(np.float32)
    return x, y, rot


def overflow_bound(env, rays, kernel):
    """the most rays one launch can queue if no CTA's queue overflows: sum over tiles of min(tile rays, capacity)"""
    return sum(min(int(c) * rays, PEND_CAP[kernel]) for c in env.debug_tiles()[:, 1])


@pytest.mark.parametrize("kernel,rays,n,tile,ticks,knobs", [
    ("staged", 32, 1024, 512, 20, {"OK_BEAM_BATCH_AGENTS": 512}),  # 16,384 rays a tile; one warp-wide min per 32 rays
    ("staged", 257, 510, 255, 12, {}),                              # 65,535 rays a tile (16-bit bound); per-lane min
    ("unstaged", 1024, 300, 3, 10, {}),                             # 3,072 rays a tile
])
def test_full_ray_queue(monkeypatch, kernel, rays, n, tile, ticks, knobs):
    """Every agent off the lane, in no covered cell: pass A queues all its rays, far more than the CTA's queue holds, and
    the overflow is finished in pass A.  The cast and the random ticks that follow (auto-reset puts the crashed agents
    back on the lane) against the oracle."""
    force(monkeypatch, OK_BEAM_KERNEL=kernel, OK_BEAM_TAIL=0, **knobs)
    env, ora, tid = make_pair(["Monza", "Spa"], n, rays, reward_mode=ok.REWARD_CMAES_PROGRESS, auto_reset=1)
    ora.set_threads(ora.max_threads())
    assert env.launch_stats().block_threads == BLOCK[kernel]
    counts = env.debug_tiles()[:, 1]
    assert (counts == tile).all() and tile * rays > PEND_CAP[kernel], counts
    pts = spread_points(ora, tid)
    env.reset(None, pts)
    ora.reset(None, pts)
    x, y, rot = off_lane_poses(env, tid, np.random.default_rng(rays))
    for name, v in (("pos_x", x), ("pos_y", y), ("rot", rot), ("crashed", np.zeros(n, np.uint8))):
        env.write(name, v)
        ora.buffer(name)[:] = v
    env.debug_stats(True)
    env.cast_rays()
    ora.cast_rays()
    cast, queued, _ = env.debug_stats(True)
    assert cast == n * rays and queued == cast, (cast, queued)  # no origin covered: every ray queued
    assert queued > overflow_bound(env, rays, kernel), "no CTA's queue overflowed"
    assert_same(env, ora, ctx="cast")
    assert (env.read("hit_seg") >= 0).mean() > 0.25, "too few walls within range"
    for step in range(ticks):
        step_pair(env, ora, step)
        if step == 0:
            _, queued, _ = env.debug_stats(True)
            assert queued > overflow_bound(env, rays, kernel), "no queue overflowed in the moving tick"
        if step % 4 == 0 or step == ticks - 1:
            assert_same(env, ora, ctx=f"tick {step}")
    env.debug_stats(False)
    no_violations(env)


# ---------------------------------------------------------------------------------------------------------------------
# B. phase 4 with one thread per agent
# ---------------------------------------------------------------------------------------------------------------------
VARIANTS = {  # reset-draw flags, lap target (None = accounting off), reward mode
    "plain": (0, None, ok.REWARD_CMAES_PROGRESS),
    "drawn": (7, None, ok.REWARD_LANE_CENTER),
    "laps": (7, 2, ok.REWARD_Q_PROGRESS),
}


@pytest.mark.parametrize("variant", list(VARIANTS))
def test_one_thread_per_agent_phase4(monkeypatch, variant):
    """Staged tiles of 600 agents (phase 4 with agent_post<1> and the one-lane window search) next to tiles of 300 (two
    lanes), in the plain, drawn and laps kernels.  Every 7th agent is teleported by up to 300 px mid-run, so the window
    search around its last index cannot prove its result and the warp's full search takes over."""
    force(monkeypatch, OK_BEAM_KERNEL="staged", OK_BEAM_TAIL=0, OK_BEAM_BATCH_AGENTS=600)
    draws, target, reward = VARIANTS[variant]
    n, rays, ticks, teleport_at = 1800, 16, 90, 30
    env, ora, tid = make_pair(["IMS", "Oschersleben"], n, rays, reward_mode=reward, auto_reset=1)
    ora.set_threads(ora.max_threads())
    assert env.launch_stats().block_threads == 1024
    counts = env.debug_tiles()[:, 1]
    # the shared memory behind these two tracks holds 600 agent records: the tiles are the batch, not less
    assert sorted(counts.tolist()) == [300, 300, 600, 600], counts
    env.set_reset_draw_flags(SEED, draws)
    drawn = DrawnResets(ora, SEED, draws)
    laps = Laps(ora, drawn)
    pts = spread_points(ora, tid)
    env.reset(None, pts)
    laps.reset(None, pts)
    if target is not None:
        env.set_laps(target)
        laps.set(True, target)
        plant(laps, env, np.random.default_rng(11))
    rng = np.random.default_rng(3)
    lap_events = completions = 0
    for step in range(ticks):
        if step == teleport_at:
            x, y = ora.buffer("pos_x").copy(), ora.buffer("pos_y").copy()
            x[::7] += rng.uniform(-300, 300, size=x[::7].shape).astype(np.float32)
            y[::7] += rng.uniform(-300, 300, size=y[::7].shape).astype(np.float32)
            env.write("pos_x", x), env.write("pos_y", y)
            ora.buffer("pos_x")[:] = x
            ora.buffer("pos_y")[:] = y
        env.launch_steps_random(step, 1)
        ora.fill_random_actions(step)
        before = laps.s["laps"].copy()
        laps.step()
        lap_events += int(np.sum(laps.s["laps"] > before))
        completions += int(laps.s["completed"].sum())
        if step % 15 == 14:
            assert_same(env, ora, ctx=f"{variant}, tick {step}")
            if target is not None:
                assert_laps(env, laps, f"{variant}, tick {step}")
    if draws:
        assert drawn.k.sum() > 0, "no drawn reset happened"
    if target is not None:
        assert lap_events > 0 and completions > 0, "no lap or no completion"
    no_violations(env)


def test_balanced_tiles_above_512_against_oracle_slices():
    """The library's own balanced tiling of the bench workload at 84,000 agents: one wave of 148 tiles of about 570 agents
    (the shared memory behind all 23 tracks holds 616), before and after the re-balancing from measured tile times.  Four
    64-agent slices inside such tiles are shadowed by the oracle for 300 ticks, every buffer compared every 50."""
    n = 84000
    env = ok.Env(device=0, movement_mode=ok.MOVE_VELOCITY, reward_mode=ok.REWARD_CMAES_PROGRESS, auto_reset=1)
    bench.build_workload(ok, env, n)
    assert env.launch_stats().block_threads == 1024
    first = env.debug_tiles()
    big = first[first[:, 1] > 512]
    assert len(big) >= 4, first[:, 1].max()
    pick = big[np.linspace(0, len(big) - 1, 4).astype(int)]
    starts = [int(b) + (int(c) - 64) // 2 for _, c, b in pick]
    oracles = [_oracle_slice(lo, 64, n) for lo in starts]
    for t0 in range(0, 300, 50):
        env.launch_steps_random(t0, 50, bench.SEED)
        for ora in oracles:
            for s in range(t0, t0 + 50):
                ora.fill_random_actions(s, bench.SEED)
                ora.step()
        env.sync()
        for lo, ora in zip(starts, oracles):
            for name in ALL_BUFS:
                got, want = env.read(name)[lo:lo + 64], ora.buffer(name)
                assert same_bits(got, want).all(), f"tick {t0 + 50}, agents {lo}..{lo + 63}, buffer {name}"
    after = env.debug_tiles()
    assert not np.array_equal(after, first), "the tiling was never re-balanced"
    assert (after[:, 1] > 512).any(), "no tile above 512 agents after the re-balancing"
    assert sum(int((ora.buffer("reset_pt") >= 0).sum()) for ora in oracles) > 0
    no_violations(env)


# ---------------------------------------------------------------------------------------------------------------------
# C. ray counts
# ---------------------------------------------------------------------------------------------------------------------
STAGED_RAYS = {  # rays: (tracks, agents)
    1: (["Monza", "Spa"], 1200),
    5: (["Monza", "Spa"], 1200),
    15: (["Monza", "Spa"], 1000),
    33: (["Monza", "Spa"], 600),
    48: (["Monza", "Spa"], 400),
    100: (["Monza", "Spa"], 300),
    257: (["Monza"], 300),
    1024: (["Monza"], 80),
}


@pytest.mark.parametrize("rays", list(STAGED_RAYS))
def test_staged_kernel_ray_counts(monkeypatch, rays):
    """The staged kernel at ray counts that do and do not fill warps, up to the 16-bit tile bound (65,535 // rays agents a
    tile at 257 and 1,024 rays), with guided tiles of the size the sizing picks"""
    force(monkeypatch, OK_BEAM_KERNEL="staged", OK_BEAM_TAIL=0)
    names, n = STAGED_RAYS[rays]
    env, ora, tid = make_pair(names, n, rays, reward_mode=ok.REWARD_MIN_RAY, auto_reset=1)
    ora.set_threads(ora.max_threads())
    assert env.launch_stats().block_threads == 1024
    counts = env.debug_tiles()[:, 1]
    if rays > 256:  # the tile bound, not the shared memory, sizes the tiles
        assert counts.tolist() == guided_counts(tid, 65535 // rays), counts
    else:  # each track's agents in one tile
        assert counts.tolist() == guided_counts(tid, n // len(names)), counts
    pts = spread_points(ora, tid)
    env.reset(None, pts)
    ora.reset(None, pts)
    for step in range(25):
        step_pair(env, ora, step)
        if step % 8 == 0 or step == 24:
            assert_same(env, ora, ctx=f"{rays} rays, tick {step}")
    assert (ora.buffer("reset_pt") != pts).any(), "nobody crashed: test too weak"
    no_violations(env)


GRID_RAYS = {1: 300, 33: 200, 257: 48, 1024: 16}  # rays: agents


@pytest.mark.parametrize("raycast", [ok.RAYCAST_GRID, ok.RAYCAST_BRUTE])
@pytest.mark.parametrize("rays", list(GRID_RAYS))
def test_grid_and_brute_ray_counts(rays, raycast):
    n = GRID_RAYS[rays]
    env, ora, tid = make_pair(["Monza", "Spa"], n, rays, raycast_mode=raycast, reward_mode=ok.REWARD_MIN_RAY, auto_reset=1)
    ora.set_threads(ora.max_threads())
    st = env.launch_stats()
    assert st.block_threads == 1024 and st.tiles > 0 and len(env.debug_tiles()) == 0, "not the grid kernel's tiling"
    pts = spread_points(ora, tid)
    env.reset(None, pts)
    ora.reset(None, pts)
    for step in range(25):
        step_pair(env, ora, step)
        if step % 8 == 0 or step == 24:
            assert_same(env, ora, ctx=f"{rays} rays, mode {raycast}, tick {step}")
    no_violations(env)


# ---------------------------------------------------------------------------------------------------------------------
# D. ok_lidar_query's three mappings
# ---------------------------------------------------------------------------------------------------------------------
def lidar_mapping(rays):
    """the query kernel's thread mapping for a fan of `rays` (lidar_threads_per_pose, ok_lidar_query.cuh:34-42)"""
    if rays <= 32:
        return "poses per warp"
    return "warp groups" if rays <= 256 else "one pose per CTA, looping"


QUERY_RAYS = [1, 17, 31, 32, 64, 100, 256, 257, 1000, 1024]
assert {lidar_mapping(r) for r in QUERY_RAYS} == {"poses per warp", "warp groups", "one pose per CTA, looping"}


@pytest.mark.parametrize("rays", QUERY_RAYS)
def test_lidar_query_mappings(rays):
    """Hard poses on four tracks, each ray count in beam, grid and brute-force mode: the query equals ok_cast_rays of agents
    at the same poses with that fan, on every output; at 100, 257 and 1,024 rays it also equals the oracle."""
    names = ["Monza", "Spa", "Oschersleben", "Austin"]
    cfg = dict(sensor_range=137.5, sensor_offset=3.25)
    env = ok.Env(device=0, **cfg)
    for nm in names:
        env.add_named_track(nm)
    rng = np.random.default_rng(1000 + rays)
    n = 420
    x, y, rot, tid = _hard_poses(env, rng, n, len(names))
    fan = np.sort(rng.uniform(-100.0, 100.0, rays)).astype(np.float32)
    env.alloc_agents(n, fan, tid)
    ora = None
    if rays in (100, 257, 1024):
        ora = Oracle("port", **cfg)
        for nm in names:
            ora.add_track(ok.track_columns(nm))
        ora.alloc_agents(n, fan, tid)
        ora.set_threads(ora.max_threads())
        ora.buffer("pos_x")[:], ora.buffer("pos_y")[:], ora.buffer("rot")[:] = x, y, rot
        ora.buffer("crashed")[:] = 0
        ora.cast_rays()
    for mode in ("beam", "grid", "brute"):
        env.update_config(raycast_mode=MODES[mode])
        for name, v in (("pos_x", x), ("pos_y", y), ("rot", rot), ("crashed", np.zeros(n, np.uint8))):
            env.write(name, v)
        env.cast_rays()
        launches = env.launch_stats().kernel_launches
        got = env.lidar_query(x, y, rot, tid, fan)
        assert env.launch_stats().kernel_launches == launches + 1
        for nm in NAMES:
            want = env.read(C_NAMES[nm])
            assert got[nm].shape == want.shape, (mode, nm)
            bad = np.argwhere(~same_bits(got[nm], want))
            assert len(bad) == 0, (mode, nm, "agent path", len(bad), tuple(bad[0]))
            if ora is not None:
                bad = np.argwhere(~same_bits(got[nm], ora.buffer(C_NAMES[nm])))
                assert len(bad) == 0, (mode, nm, "oracle", len(bad), tuple(bad[0]))
        seg = got["hit_seg"]
        assert (seg >= 0).any() and (seg < 0).any(), "degenerate: all hits or all misses"
    no_violations(env)
    env.close()

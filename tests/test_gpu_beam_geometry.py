"""GPU: the beam kernels and ok_lidar_query on every kind of beam table OkConfig accepts, not only the default 2 px x 256
bins.  Coarse cells and few bins give long rest lists (pass B's dealing over many 32-chunk rounds), entries flagged complete
and, with the device builder, lists that overflowed its 256-candidate scratch (no candidates, d = 0: every ray is finished
by the grid walk); fine cells and 1,024 bins give short lists and the narrowest bins, where a ray angle close to the
table's +-100 rad limit has the least headroom.  A folded synthetic track makes the host builder cut lists at 1,024
candidates.  Every comparison is bit for bit, NaN equal to NaN, against the port oracle, the brute-force ray cast or the
agent path, and every test first asserts from the env's own tables (beam_lookup_ex) and counters (debug_stats) that it
runs the path it is named for."""
import math

import numpy as np
import pytest

import openkitchen_b200 as ok
from oracle.api import Oracle
from tests.test_beam_geometry_cpu import FOLD_POINTS, MAX_LIST, folded_track
from tests.test_gpu_lidar_query import C_NAMES, MODES, NAMES, _hard_poses
from tests.util import ALL_BUFS, RAY_BUFS, assert_same, make_pair, same_bits, spread_points

pytestmark = pytest.mark.gpu

TRACKS = ["Spa", "Zandvoort", "Monza"]
GEOMETRIES = [(2.0, 128), (4.0, 128), (1.5, 64), (8.0, 32), (16.0, 16), (64.0, 8), (32.0, 8), (64.0, 1024), (2.0, 1024)]
RB = 201.0  # completeness distance of an entry flagged complete: Agent::kSensorRange + 1 (BeamConfig, beam_plan)
DEG2RAD = np.float32(0.0174532924)  # OK_DEG2RAD
MAX_ANGLE = 100.0  # kBeamMaxAngle: rays with a larger |angle| (rad) skip the table


def coarse(cell):
    """the geometries where the two builders produce different tables (the device builder's lists overflow)"""
    return cell >= 8.0


def use_builder(monkeypatch, builder, kernel=None):
    """one builder for this test, no disk cache, and no table another test built (the in-process cache is keyed on the
    geometry, not on the builder)"""
    monkeypatch.setenv("OK_BEAM_CACHE", "0")
    monkeypatch.setenv("OK_BEAM_BUILDER", builder)
    if kernel:
        monkeypatch.setenv("OK_BEAM_KERNEL", kernel)
    ok.release_caches()


def no_violations(env):
    n, _ = env.debug_violations()
    assert n == 0, f"{n} out-of-range indices counted"


def ray_angles(rot, fan):
    """per (agent, ray) the angle the kernels look the table up with: fmul(OK_DEG2RAD, fadd(rot, ray_deg))"""
    return ((np.asarray(rot, np.float32)[:, None] + np.asarray(fan, np.float32)[None, :]).astype(np.float32) * DEG2RAD).astype(np.float32)


def table_paths(env, tid, x, y, ang, limit=None, rng=None):
    """what the env's own tables hold for these rays (origin = x, y; sensor offset 0): counts of covered rays, of rays whose
    entry overflowed in the device builder (no candidate, d = 0), whose list was cut (MAX_LIST candidates), whose rest has
    more than 32 / 100 chunks, whose entry is flagged complete, and of rays within 0.1 rad below the angle limit"""
    pairs = [(a, r) for a in range(ang.shape[0]) for r in range(ang.shape[1])]
    if limit is not None and len(pairs) > limit:
        pairs = [pairs[i] for i in rng.choice(len(pairs), limit, replace=False)]
    c = dict(covered=0, overflow=0, cut=0, rest32=0, rest100=0, complete=0, near_limit=0, max_rest=0)
    for a, r in pairs:
        got = env.beam_lookup_ex(int(tid[a]), float(x[a]), float(y[a]), float(ang[a, r]))
        if got is None:
            continue
        items, d, _, _ = got
        rest = (max(len(items) - 4, 0) + 3) // 4
        c["covered"] += 1
        c["overflow"] += len(items) == 0 and d == 0.0
        c["cut"] += len(items) == MAX_LIST
        c["rest32"] += rest > 32
        c["rest100"] += rest > 100
        c["complete"] += d == RB
        c["near_limit"] += abs(float(ang[a, r])) > MAX_ANGLE - 0.1
        c["max_rest"] = max(c["max_rest"], rest)
    return c


def step_pair(env, ora, step):
    env.launch_steps_random(step, 1)
    ora.fill_random_actions(step)
    ora.step()


# ---------------------------------------------------------------------------------------------------------------------
# 1. rollouts against the oracle, per geometry, kernel shape and builder
# ---------------------------------------------------------------------------------------------------------------------
ROLLOUTS = [(cell, bins, builder) for cell, bins in GEOMETRIES for builder in (("gpu", "cpu") if coarse(cell) else ("gpu",))]


@pytest.mark.parametrize("kernel", ["staged", "unstaged"])
@pytest.mark.parametrize("cell,bins,builder", ROLLOUTS)
def test_rollout_parity_per_geometry(monkeypatch, cell, bins, builder, kernel):
    """Spa, Zandvoort and Monza with auto-reset and the reward that reads min_dist2, at 32 and 45 rays: 40 random ticks,
    every buffer equal to the oracle.  The rays of the first cast must meet the entries this geometry is about: at 32 px
    cells and above lists flagged complete, and at 8 bins either lists of more than 100 rest chunks (host builder) or
    overflowed lists (device builder)."""
    use_builder(monkeypatch, builder, kernel)
    queued = walked = 0
    for rays in (32, 45):
        env, ora, tid = make_pair(TRACKS, 3 * 64, rays, raycast_mode=ok.RAYCAST_BEAM, beam_cell=cell, beam_bins=bins,
                                  reward_mode=ok.REWARD_MIN_RAY, auto_reset=1)
        ora.set_threads(ora.max_threads())
        assert env.launch_stats().block_threads == (1024 if kernel == "staged" else 256)
        pts = spread_points(ora, tid)
        env.reset(None, pts)
        ora.reset(None, pts)
        paths = table_paths(env, tid, env.read("pos_x"), env.read("pos_y"), ray_angles(env.read("rot"), ok.ray_fan(rays)))
        assert paths["covered"] > 0.9 * 3 * 64 * rays, paths
        if cell >= 32.0:
            assert paths["complete"] > 0, paths
        if bins == 8:
            if builder == "cpu":
                assert paths["rest100"] > 0, paths
            else:
                assert paths["overflow"] > 0 and paths["max_rest"] <= 63, paths  # 256-candidate scratch: <= 63 chunks
        env.debug_stats(True)
        for step in range(40):
            step_pair(env, ora, step)
            if step % 10 == 9:
                assert_same(env, ora, ctx=f"{cell} px x {bins} bins, {builder} builder, {kernel}, {rays} rays, tick {step}")
        _, q, w = env.debug_stats(False)
        queued, walked = queued + q, walked + w
        assert (ora.buffer("reset_pt") != pts).any(), "nobody crashed: test too weak"
        no_violations(env)
        env.close()
    assert queued > 0, "no ray went to pass B"
    if coarse(cell):
        assert walked > 0, "no ray was finished by the grid walk"


def test_device_builder_reports_overflowed_lists(monkeypatch, capfd):
    """A one-track env at 64 px x 8 bins on Spa: the device builder counts lists longer than its scratch in its verbose
    line, and they reach the table as entries with no candidate and d = 0"""
    use_builder(monkeypatch, "gpu")
    monkeypatch.setenv("OK_BEAM_VERBOSE", "1")
    env = ok.Env(device=0, beam_cell=64.0, beam_bins=8)
    t = env.add_named_track("Spa")
    env.alloc_agents(1, ok.ray_fan(1), np.zeros(1, np.int32))
    line = [ln for ln in capfd.readouterr().err.splitlines() if ln.startswith("[ok_beam_gpu] rows")]
    assert len(line) == 1, line
    assert int(line[0].split(", ")[-1].split()[0]) > 0, line[0]
    x, y = env.track_array(t, "x"), env.track_array(t, "y")
    empty = [env.beam_lookup_ex(t, float(x[i]), float(y[i]), float(a)) for i in range(0, len(x), 7) for a in (-2.5, 0.3, 1.9)]
    assert any(g is not None and len(g[0]) == 0 and g[1] == 0.0 for g in empty)
    env.close()


# ---------------------------------------------------------------------------------------------------------------------
# 2. beam mode against brute force, with ray angles at the table's limit
# ---------------------------------------------------------------------------------------------------------------------
def near_limit_rot(rng, n):
    """headings that put the middle rays of the -70..70 degree fan within a few degrees of +-100 rad, on both sides"""
    limit = MAX_ANGLE * 180.0 / math.pi
    return (np.where(rng.random(n) < 0.5, -1.0, 1.0) * limit + rng.uniform(-4.0, 4.0, n)).astype(np.float32)


@pytest.mark.parametrize("cell,bins,builder", [(64.0, 8, "cpu"), (64.0, 8, "gpu"), (8.0, 32, "cpu"), (2.0, 1024, "gpu"),
                                               (64.0, 1024, "cpu")])
def test_beam_equals_brute_force_near_the_angle_limit(monkeypatch, cell, bins, builder):
    """Twin populations at the same poses, one in beam mode and one in brute-force mode; a third of the agents head within
    4 degrees of +-100 rad.  The cast and 25 ticks after it: every ray buffer, and every other buffer, bit-equal."""
    use_builder(monkeypatch, builder)
    n, rays = 3 * 64, 32
    cfg = dict(beam_cell=cell, beam_bins=bins, reward_mode=ok.REWARD_MIN_RAY, auto_reset=1)
    beam, _, tid = make_pair(TRACKS, n, rays, raycast_mode=ok.RAYCAST_BEAM, **cfg)
    brute, ora, _ = make_pair(TRACKS, n, rays, raycast_mode=ok.RAYCAST_BRUTE, **cfg)
    pts = spread_points(ora, tid)
    rng = np.random.default_rng(int(cell) * 4096 + bins)
    beam.reset(None, pts)
    brute.reset(None, pts)
    rot = beam.read("rot")
    rot[::3] = near_limit_rot(rng, len(rot[::3]))
    for e in (beam, brute):
        e.write("rot", rot)
        e.cast_rays()
    x, y = beam.read("pos_x"), beam.read("pos_y")
    ang = ray_angles(rot, ok.ray_fan(rays))
    paths = table_paths(beam, tid, x, y, ang)
    assert paths["near_limit"] > 0, paths  # covered rays within 0.1 rad below the limit
    assert (np.abs(ang) >= MAX_ANGLE).any() and (np.abs(ang[::3]) < MAX_ANGLE).any()
    ctx = f"{cell} px x {bins} bins, {builder} builder"
    for name in ALL_BUFS:
        assert same_bits(beam.read(name), brute.read(name)).all(), f"{ctx}, cast: {name}"
    beam.debug_stats(True)
    for step in range(25):
        beam.launch_steps_random(step, 1)
        brute.launch_steps_random(step, 1)
        if step % 5 == 4:
            for name in ALL_BUFS:
                assert same_bits(beam.read(name), brute.read(name)).all(), f"{ctx}, tick {step}: {name}"
    _, queued, _ = beam.debug_stats(False)
    assert queued > 0
    no_violations(beam)


# ---------------------------------------------------------------------------------------------------------------------
# 3. ok_lidar_query in beam mode, in its three thread mappings
# ---------------------------------------------------------------------------------------------------------------------
QUERY_GEOMETRIES = [(64.0, 8, "cpu"), (64.0, 8, "gpu"), (32.0, 8, "cpu"), (16.0, 16, "gpu"), (64.0, 1024, "cpu"),
                    (2.0, 1024, "gpu")]


@pytest.mark.parametrize("rays", [31, 200, 700])  # poses per warp / warp groups / one pose per CTA, looping
@pytest.mark.parametrize("cell,bins,builder", QUERY_GEOMETRIES)
def test_lidar_query_per_geometry(monkeypatch, cell, bins, builder, rays):
    """Hard poses (and headings at the angle limit) on three tracks: the beam-mode query equals ok_cast_rays of agents at
    the same poses, and the brute-force query, on every output"""
    use_builder(monkeypatch, builder)
    env = ok.Env(device=0, raycast_mode=ok.RAYCAST_BEAM, beam_cell=cell, beam_bins=bins)
    for nm in TRACKS:
        env.add_named_track(nm)
    rng = np.random.default_rng(rays + int(cell) * bins)
    n = 300
    x, y, rot, tid = _hard_poses(env, rng, n, len(TRACKS))
    rot[1::4] = near_limit_rot(rng, len(rot[1::4]))
    fan = np.sort(rng.uniform(-100.0, 100.0, rays)).astype(np.float32)
    env.alloc_agents(n, fan, tid)
    fin = np.isfinite(x) & np.isfinite(y) & np.isfinite(rot)
    paths = table_paths(env, tid, np.where(fin, x, 0), np.where(fin, y, 0), ray_angles(np.where(fin, rot, 0), fan), 4000, rng)
    assert paths["covered"] > 500, paths
    if bins == 8 and builder == "cpu":
        assert paths["rest32"] > 0, paths  # a ray alone has more chunks than one round deals
    if bins == 1024:
        assert paths["near_limit"] > 0, paths
    for name, v in (("pos_x", x), ("pos_y", y), ("rot", rot), ("crashed", np.zeros(n, np.uint8))):
        env.write(name, v)
    env.cast_rays()
    beam = env.lidar_query(x, y, rot, tid, fan)
    for nm in NAMES:
        bad = np.argwhere(~same_bits(beam[nm], env.read(C_NAMES[nm])))
        assert len(bad) == 0, (nm, "agent path", len(bad), tuple(bad[0]))
    env.update_config(raycast_mode=MODES["brute"])
    brute = env.lidar_query(x, y, rot, tid, fan)
    for nm in NAMES:
        bad = np.argwhere(~same_bits(beam[nm], brute[nm]))
        assert len(bad) == 0, (nm, "brute force", len(bad), tuple(bad[0]))
    seg = beam["hit_seg"]
    assert (seg >= 0).any() and (seg < 0).any()
    no_violations(env)
    env.close()


# ---------------------------------------------------------------------------------------------------------------------
# 4. lists cut by the host builder (and overflowed in the device builder) on a folded track
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kernel", ["staged", "unstaged"])
@pytest.mark.parametrize("builder", ["cpu", "gpu"])
def test_folded_track_parity(monkeypatch, builder, kernel):
    """Agents started on the folded stretch of tests/test_beam_geometry_cpu.py's synthetic track at 64 px x 8 bins, next
    to Monza: their rays start in cells whose lists the host builder cuts at 1,024 candidates (the device builder's
    overflow instead).  The cast and 30 random ticks against the oracle."""
    use_builder(monkeypatch, builder, kernel)
    n, rays = 256, 32
    cfg = dict(reward_mode=ok.REWARD_MIN_RAY, auto_reset=1)
    tid = (np.arange(n) >= n // 2).astype(np.int32)
    env = ok.Env(device=0, raycast_mode=ok.RAYCAST_BEAM, beam_cell=64.0, beam_bins=8, **cfg)
    ora = Oracle("port", **cfg)
    for cols in (folded_track(), ok.track_columns("Monza")):
        env.add_track(cols)
        ora.add_track(cols)
    fan = ok.ray_fan(rays)
    env.alloc_agents(n, fan, tid)
    ora.alloc_agents(n, fan, tid)
    ora.set_threads(ora.max_threads())
    pts = spread_points(ora, tid)
    pts[: n // 2] = np.linspace(0, FOLD_POINTS - 1, n // 2).astype(np.int32)
    env.reset(None, pts)
    ora.reset(None, pts)
    paths = table_paths(env, tid, env.read("pos_x"), env.read("pos_y"), ray_angles(env.read("rot"), fan))
    assert paths[{"cpu": "cut", "gpu": "overflow"}[builder]] > 100, paths
    env.debug_stats(True)
    env.cast_rays()
    ora.cast_rays()
    assert_same(env, ora, names=RAY_BUFS, ctx=f"{builder} builder, {kernel}, cast")
    for step in range(30):
        step_pair(env, ora, step)
        if step % 10 == 9:
            assert_same(env, ora, ctx=f"{builder} builder, {kernel}, tick {step}")
    _, queued, walked = env.debug_stats(False)
    assert queued > 0 and walked > 0, (queued, walked)
    no_violations(env)
    env.close()


# ---------------------------------------------------------------------------------------------------------------------
# 5. a geometry whose table cannot be built
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("builder", ["auto", "gpu", "cpu"])
def test_geometry_too_large_is_a_clean_error(monkeypatch, builder):
    """1 px x 1,024 bins on Zandvoort: ok_alloc_agents fails with OK_ERR_INVALID_ARG and "beam table too large", with
    either builder and none forced.  A default env in the same process then builds and matches the oracle."""
    use_builder(monkeypatch, builder)
    env = ok.Env(device=0, raycast_mode=ok.RAYCAST_BEAM, beam_cell=1.0, beam_bins=1024)
    env.add_named_track("Zandvoort")
    with pytest.raises(ok.OkError) as err:
        env.alloc_agents(64, ok.ray_fan(32), np.zeros(64, np.int32))
    assert err.value.code == -1 and "beam table too large" in str(err.value), str(err.value)
    env.close()
    env, ora, tid = make_pair(["Zandvoort", "Monza"], 128, 32, reward_mode=ok.REWARD_CMAES_PROGRESS, auto_reset=1)
    pts = spread_points(ora, tid)
    env.reset(None, pts)
    ora.reset(None, pts)
    for step in range(20):
        step_pair(env, ora, step)
    assert_same(env, ora, ctx="default env after the failed build")
    no_violations(env)
    env.close()

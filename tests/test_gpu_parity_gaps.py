"""GPU parity, second file: the cases round 1 left open -- non-default constants (sensor offset, dt, crash threshold,
standstill window, speed limit) in all three narrow phases, the north star's 1,000 ticks at the full C3 shape against
oracle slices, sharded == unsharded through OkConfig::agent_id_base, and the reference's REAL CUDA kernel on all 23
tracks with the hit segment recovered from its hit points."""
import ctypes as C
import os

import numpy as np
import pytest

import bench
import openkitchen_b200 as ok
from oracle.api import Oracle, have_ref
from tests.util import ALL_BUFS, assert_same, make_pair, same_bits, spread_points

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB_CUDA = os.path.join(ROOT, "oracle", "_ref", "libokref_cuda.so")
RAYCASTS = [ok.RAYCAST_BEAM, ok.RAYCAST_GRID, ok.RAYCAST_BRUTE]


@pytest.mark.parametrize("raycast", RAYCASTS)
@pytest.mark.parametrize("offset", [3.0, -5.0, 17.5])
def test_sensor_offset(raycast, offset):
    """Agent::sensor_offset_ != 0 (CollisionChecker.cu:121-124): the lidar origin leaves the agent's position, which is
    what the beam-table row lookup and the hit rotation are keyed on."""
    env, ora, tid = make_pair(["Monza", "Sepang", "Spa"], 96, 32, raycast_mode=raycast, sensor_offset=offset,
                              reward_mode=ok.REWARD_MIN_RAY, auto_reset=1)
    pts = spread_points(ora, tid)
    env.reset(None, pts)
    ora.reset(None, pts)
    for step in range(80):
        env.launch_steps_random(step, 1)
        ora.fill_random_actions(step)
        ora.step()
        if step % 20 == 0:
            assert_same(env, ora, ctx=f"sensor_offset {offset} step {step}")
    assert_same(env, ora, ctx=f"sensor_offset {offset}")
    assert not np.array_equal(env.read("hit_abs")[:, 0] - env.read("hit_rel")[:, 0], 0), "degenerate"


@pytest.mark.parametrize("raycast", RAYCASTS)
@pytest.mark.parametrize("mode", [ok.MOVE_VELOCITY, ok.MOVE_ACCELERATION])
def test_non_default_constants(raycast, mode):
    """dt, collision threshold, standstill window / threshold, speed limit, sensor range, auto-reset stride: none at
    the reference's value (Agent.h:10-12, Agent.cpp:84,110, Environment.h:19-20, CollisionChecker.cu:167)"""
    env, ora, tid = make_pair(["Austin", "Budapest", "Zandvoort", "Melbourne"], 128, 15, raycast_mode=raycast,
                              movement_mode=mode, reward_mode=ok.REWARD_CMAES_PROGRESS, auto_reset=1, auto_reset_stride=41,
                              dt=0.021, collision_dist2=9.5, standstill_period=37, standstill_threshold=31.0,
                              speed_limit=23.0, sensor_range=150.0, sensor_offset=1.25)
    pts = spread_points(ora, tid)
    env.reset(None, pts)
    ora.reset(None, pts)
    for step in range(160):
        env.launch_steps_random(step, 1)
        ora.fill_random_actions(step)
        ora.step()
        if step % 40 == 39:
            assert_same(env, ora, ctx=f"constants step {step}")
    assert ora.buffer("timed_out").any() or (ora.buffer("reset_pt") != pts).any(), "nothing ever crashed: test too weak"
    if mode == ok.MOVE_ACCELERATION:
        assert float(ora.buffer("speed").max()) <= 23.0


def test_update_config_mid_rollout():
    """the per-tick constants can change on a live env (ok_update_config) and take effect on the next tick"""
    env, ora, tid = make_pair(["Sochi"], 64, 32, reward_mode=ok.REWARD_Q_PROGRESS, auto_reset=1)
    pts = spread_points(ora, tid)
    env.reset(None, pts)
    ora.reset(None, pts)
    for step in range(90):
        if step == 30:
            env.update_config(sensor_offset=-2.0, dt=0.01, collision_dist2=4.0)
            ora.cfg.sensor_offset, ora.cfg.dt, ora.cfg.collision_dist2 = -2.0, 0.01, 4.0
            ora.update_config()
        if step == 60:
            env.update_config(movement_mode=ok.MOVE_ACCELERATION, speed_limit=40.0)
            ora.cfg.movement_mode, ora.cfg.speed_limit = 1, 40.0
            ora.update_config()
        env.launch_steps_random(step, 1)
        ora.fill_random_actions(step)
        ora.step()
    assert_same(env, ora, ctx="update_config")


def _oracle_slice(lo, count, n_total, kind="port"):
    """the agents [lo, lo + count) of the bench workload (bench.build_workload) alone in an oracle"""
    names = ok.track_names()
    ora = Oracle(kind, movement_mode=0, reward_mode=2, auto_reset=1, agent_id_base=lo)
    pts_per = []
    for nm in names:
        cols = ok.track_columns(nm)
        ora.add_track(cols)
        pts_per.append(len(cols[0]))
    ids = np.arange(lo, lo + count, dtype=np.int64)
    tid = (ids * len(names) // n_total).astype(np.int32)
    ora.alloc_agents(count, ok.ray_fan(32), tid)
    pts = ((ids.astype(np.uint64) * np.uint64(2654435761)) % np.uint64(2**32) % np.asarray(pts_per, dtype=np.uint64)[tid]).astype(np.int32)
    ora.reset(None, pts)
    ora.set_threads(ora.max_threads())
    return ora


def test_c3_shape_1000_ticks_against_oracle_slices():
    """North star: 1,000 steps.  The full C3 batch (65,536 agents x 23 tracks x 32 rays, Philox actions generated in
    the kernel, auto-reset) runs 1,000 ticks; four 64-agent slices of it (256 agents, on four different tracks) are
    shadowed by the oracle -- agents are independent, so each slice must evolve exactly like the same agents alone --
    and every buffer is compared bit for bit every 100 ticks."""
    n = 65536
    env = ok.Env(device=0, movement_mode=ok.MOVE_VELOCITY, reward_mode=ok.REWARD_CMAES_PROGRESS, auto_reset=1)
    bench.build_workload(ok, env, n)
    starts = [0, 20000, 41111, n - 64]
    oracles = [_oracle_slice(lo, 64, n) for lo in starts]
    for t0 in range(0, 1000, 100):
        env.launch_steps_random(t0, 100, bench.SEED)
        for ora in oracles:
            for s in range(t0, t0 + 100):
                ora.fill_random_actions(s, bench.SEED)
                ora.step()
        env.sync()
        for lo, ora in zip(starts, oracles):
            for name in ALL_BUFS:
                got, want = env.read(name)[lo:lo + 64], ora.buffer(name)
                assert same_bits(got, want).all(), f"tick {t0 + 100}, agents {lo}..{lo + 63}, buffer {name}"
    resets = sum(int((ora.buffer("reset_pt") >= 0).sum()) for ora in oracles)
    assert resets > 0


def test_shard_reproduces_its_slice_of_the_unsharded_run():
    """OkConfig::agent_id_base: a rank that owns agents [lo, lo + m) of a population reproduces, bit for bit, what the
    unsharded population computes for them (same Philox stream, same reset points)."""
    n, lo, m, ticks = 8192, 4096 + 123, 1500, 60
    names = ok.track_names()
    full = ok.Env(device=0, reward_mode=ok.REWARD_CMAES_PROGRESS, auto_reset=1)
    bench.build_workload(ok, full, n)
    shard = ok.Env(device=0, reward_mode=ok.REWARD_CMAES_PROGRESS, auto_reset=1, agent_id_base=lo)
    bench.build_workload(ok, shard, m, id_base=lo, n_total=n)
    full.launch_steps_random(0, ticks, bench.SEED)
    shard.launch_steps_random(0, ticks, bench.SEED)
    full.sync(), shard.sync()
    for name in ok.BUFFERS:
        a, b = full.read(name)[lo:lo + m], shard.read(name)
        assert same_bits(a, b).all(), f"shard vs unsharded: buffer {name}"
    # and against the reference's own objects when the prebuilt checker is on the box
    if have_ref():
        ora = _oracle_slice(lo, 48, n, kind="reference")
        for s in range(ticks):
            ora.fill_random_actions(s, bench.SEED)
            ora.step()
        for name in ALL_BUFS:
            assert same_bits(shard.read(name)[:48], ora.buffer(name)).all(), f"shard vs reference objects: {name}"


def _point_segment_distance(px, py, seg):
    x1, y1, x2, y2 = (seg[..., k].astype(np.float64) for k in range(4))
    dx, dy = x2 - x1, y2 - y1
    ll = dx * dx + dy * dy
    u = np.where(ll > 0, ((px - x1) * dx + (py - y1) * dy) / np.where(ll > 0, ll, 1.0), 0.0)
    u = np.clip(u, 0.0, 1.0)
    return np.hypot(px - (x1 + u * dx), py - (y1 + u * dy))


@pytest.mark.skipif(not os.path.exists(LIB_CUDA), reason="oracle/_ref/libokref_cuda.so not built")
def test_reference_cuda_kernel_all_tracks_hit_segments(tmp_path):
    """The reference's REAL CollisionChecker / TrackSegments (CollisionChecker.cu + TrackSegments.cu compiled unchanged
    for sm_100a) on every one of the 23 tracks.  Its kernel reports hit points, not segment indices, so the index is
    recovered geometrically: the reference's hit point must lie on the segment this repo reports (CollisionChecker.cu:
    68-69 writes origin + min_t * dir).  The reference kernel uses libdevice cosf/sinf and FMA contraction, so
    distances agree to rounding (1e-4 relative, the north star's tolerance); hit / miss and crash flags must match."""
    ref = C.CDLL(LIB_CUDA)
    ref.okc_create.restype = C.c_void_p
    ref.okc_create.argtypes = [C.c_char_p, C.c_int64, C.c_int, C.c_void_p]
    ref.okc_set_poses.argtypes = [C.c_void_p] * 5
    ref.okc_check.argtypes = [C.c_void_p]
    ref.okc_get.argtypes = [C.c_void_p] * 4
    ref.okc_destroy.argtypes = [C.c_void_p]
    n, rays = 768, 32
    fan = ok.ray_fan(rays)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)
    total = off_segment = far = 0
    for name in ok.track_names():
        csv = tmp_path / f"{name}.csv"
        ok.write_track_csv(name, str(csv))
        env = ok.Env(device=0, auto_reset=1)
        t = env.add_named_track(name)
        npts = env.track_info(t).n_points
        segs = env.track_array(t, "segments")
        env.alloc_agents(n, fan)
        env.reset(None, (np.arange(n, dtype=np.int64) * 2654435761 % 2**32 % npts).astype(np.int32))
        env.launch_steps_random(0, 45)  # drive around, then freeze the poses
        env.write("crashed", np.zeros(n, dtype=np.uint8))
        env.cast_rays()
        x, y, rot = env.read("pos_x"), env.read("pos_y"), env.read("rot")
        mine_abs, mine_seg, mine_t, crashed = env.read("hit_abs"), env.read("hit_seg"), env.read("hit_t"), env.read("crashed")
        h = ref.okc_create(str(csv).encode(), n, rays, vp(fan))
        live = np.zeros(n, dtype=np.uint8)
        ref.okc_set_poses(h, vp(x), vp(y), vp(rot), vp(live))
        ref.okc_check(h)
        theirs_abs = np.zeros((n, rays, 2), dtype=np.float32)
        theirs_rel = np.zeros((n, rays, 2), dtype=np.float32)
        their_crashed = np.zeros(n, dtype=np.uint8)
        ref.okc_get(h, vp(theirs_rel), vp(theirs_abs), vp(their_crashed))
        ref.okc_destroy(h)
        env.close()
        d_theirs = np.hypot(theirs_abs[..., 0].astype(np.float64) - x[:, None], theirs_abs[..., 1].astype(np.float64) - y[:, None])
        their_hit = d_theirs < 200.0 - 1e-2
        my_hit = mine_seg >= 0
        # hit / miss: may only differ for rays that end within rounding of the sensor range
        differ = my_hit != their_hit
        assert (np.abs(mine_t[differ] - 200.0) < 5e-2).all() and (np.abs(d_theirs[differ] - 200.0) < 5e-2).all(), name
        both = my_hit & their_hit
        # the reference's hit point lies on the segment this repo reports
        dist = _point_segment_distance(theirs_abs[..., 0][both], theirs_abs[..., 1][both], segs[mine_seg[both]])
        rel = np.abs(mine_t[both] - d_theirs[both]) / np.maximum(d_theirs[both], 1e-3)
        total += int(both.sum())
        off_segment += int((dist > 2e-2).sum())
        far += int((rel > 1e-4).sum())
        near = np.abs(env_min_dist2(mine_abs, x, y) - 2.0) < 1e-3  # exactly on the crash threshold: may flip under rounding
        assert np.array_equal(crashed[~near], their_crashed[~near]), f"{name}: crash flags"
    # a ray grazing a polyline vertex can land on the neighbouring segment under different rounding: allow a handful
    assert total > 23 * n * rays * 0.5
    assert off_segment <= 2e-4 * total, f"{off_segment} of {total} reference hit points are off the reported segment"
    assert far <= 2e-4 * total, f"{far} of {total} hit distances differ by more than 1e-4 relative"


def env_min_dist2(hit_abs, x, y):
    d2 = (hit_abs[..., 0].astype(np.float64) - x[:, None]) ** 2 + (hit_abs[..., 1].astype(np.float64) - y[:, None]) ** 2
    return d2.min(axis=1)


def test_envs_of_different_sizes_interleave():
    """cudaFuncAttributeMaxDynamicSharedMemorySize belongs to the kernel, not to an env: a small env created after a
    large one must not lower the limit the large one launches with (round-1 advisor finding)"""
    big, ora_b, tid_b = make_pair(ok.track_names(), 23 * 300, 32, auto_reset=1, reward_mode=2)
    small, ora_s, tid_s = make_pair(["IMS"], 5, 7, auto_reset=1, reward_mode=2)
    for env, ora, tid in ((big, ora_b, tid_b), (small, ora_s, tid_s)):
        pts = spread_points(ora, tid)
        env.reset(None, pts)
        ora.reset(None, pts)
    for step in range(12):
        for env, ora in ((big, ora_b), (small, ora_s)):
            env.launch_steps_random(step, 1)
            ora.fill_random_actions(step)
            ora.step()
    assert_same(big, ora_b, ctx="big env")
    assert_same(small, ora_s, ctx="small env")


@pytest.mark.parametrize("flushers", [0, 6])
@pytest.mark.parametrize("n,rays", [(6000, 32), (2500, 15), (300, 32)])
def test_host_step_delivers_every_buffer(monkeypatch, n, rays, flushers):
    """ok_step_host with pinned buffers: the kernel reads the actions and writes obs / reward / done through the host
    mapping (obs as whole tiles, several tiles per CTA -- or, with OK_E2E_FLUSHERS, by flusher CTAs next to the step
    kernel that wait for a tile's flag); what arrives must be the device buffers, bit for bit, and the tiling used for
    this path must not change any result (compared with the same actions through ok_launch_step)."""
    monkeypatch.setenv("OK_E2E_FLUSHERS", str(flushers))
    names = ["Monza", "Sepang", "Spa"]
    tid = (np.arange(n) * len(names) // n).astype(np.int32)
    envs = []
    for _ in range(2):
        env = ok.Env(device=0, reward_mode=ok.REWARD_CMAES_PROGRESS, auto_reset=1)
        for nm in names:
            env.add_named_track(nm)
        env.alloc_agents(n, ok.ray_fan(rays), tid)
        envs.append(env)
    a, b = envs
    rng = np.random.default_rng(5)
    thr, steer = ok.pinned_array((n,), np.float32), ok.pinned_array((n,), np.float32)
    obs, rew, done = ok.pinned_array((n, rays), np.float32), ok.pinned_array((n,), np.float32), ok.pinned_array((n,), np.uint8)
    for step in range(30):
        thr[:] = rng.random(n, dtype=np.float32) * 100.0
        steer[:] = rng.random(n, dtype=np.float32) * 10.0 - 5.0
        obs[:], rew[:], done[:] = -1.0, -1.0, 7
        a.step_host(thr, steer, obs, rew, done)
        b.write("act_throttle", thr)
        b.write("act_steer", steer)
        b.launch_step()
        assert np.array_equal(obs.view(np.uint32), b.read("obs").view(np.uint32)), f"obs, step {step}"
        assert np.array_equal(rew.view(np.uint32), b.read("reward").view(np.uint32)), f"reward, step {step}"
        assert np.array_equal(done, b.read("done")), f"done, step {step}"
    for name in ok.BUFFERS:
        assert np.array_equal(a.read(name).view(np.uint8), b.read(name).view(np.uint8)), name
    assert (a.read("reset_pt") != 3).any() or n < 1000, "nobody ever crashed: test too weak"


@pytest.mark.parametrize("raycast", [ok.RAYCAST_BEAM, ok.RAYCAST_GRID])
@pytest.mark.parametrize("n,rays", [(6000, 32), (2500, 15), (300, 5)])
def test_host_step_q16_is_the_rounded_float_observation(n, rays, raycast):
    """ok_step_host_q16 (opt-in, lossy): what arrives is rn(clamp(obs, 0, 1) * 65535) of the SAME binary32 observation
    ok_step_host delivers -- the quantisation is the only difference, and the device state stays exact (every buffer
    compared with an env stepped through ok_launch_step on the same actions).  Whole-tile flush (rays a multiple of 8),
    the ragged fallback (15 and 5 rays) and the per-ray stores of the grid kernel."""
    names = ["Monza", "Sepang", "Spa"]
    tid = (np.arange(n) * len(names) // n).astype(np.int32)
    envs = []
    for _ in range(2):
        env = ok.Env(device=0, reward_mode=ok.REWARD_CMAES_PROGRESS, auto_reset=1, raycast_mode=raycast)
        for nm in names:
            env.add_named_track(nm)
        env.alloc_agents(n, ok.ray_fan(rays), tid)
        envs.append(env)
    a, b = envs
    rng = np.random.default_rng(6)
    thr, steer = ok.pinned_array((n,), np.float32), ok.pinned_array((n,), np.float32)
    q, rew, done = ok.pinned_array((n, rays), np.uint16), ok.pinned_array((n,), np.float32), ok.pinned_array((n,), np.uint8)
    worst = 0.0
    for step in range(20):
        thr[:] = rng.random(n, dtype=np.float32) * 100.0
        steer[:] = rng.random(n, dtype=np.float32) * 10.0 - 5.0
        q[:], rew[:], done[:] = 12345, -1.0, 7
        a.step_host(thr, steer, q, rew, done)
        b.write("act_throttle", thr)
        b.write("act_steer", steer)
        b.launch_step()
        obs = b.read("obs")
        assert np.isfinite(obs).all()
        want = ok.quantize_obs_q16(obs)
        assert np.array_equal(q, want), f"q16 obs, step {step}: {(q != want).sum()} differ"
        worst = max(worst, float(np.abs(ok.dequantize_obs_q16(q).astype(np.float64) - obs).max()))
        assert np.array_equal(rew.view(np.uint32), b.read("reward").view(np.uint32)), f"reward, step {step}"
        assert np.array_equal(done, b.read("done")), f"done, step {step}"
    assert worst <= 0.5 / 65535.0 + 2.0**-22, worst  # half a step of the fixed point + binary32 roundings (obs * 65535, q / 65535)
    for name in ok.BUFFERS:
        assert np.array_equal(a.read(name).view(np.uint8), b.read(name).view(np.uint8)), name


def test_host_step_q16_rejects_pageable_memory():
    env = ok.Env(device=0)
    env.add_named_track("Monza")
    env.alloc_agents(64, ok.ray_fan(8), np.zeros(64, np.int32))
    q = np.zeros((64, 8), np.uint16)
    with pytest.raises(ok.OkError):
        env.step_host(None, None, q, None, None)


@pytest.mark.parametrize("kernel", ["staged", "unstaged"])
@pytest.mark.parametrize("mode", [ok.MOVE_VELOCITY, ok.MOVE_ACCELERATION])
def test_both_beam_kernel_shapes_match_the_oracle(monkeypatch, kernel, mode):
    """The beam kernel has two shapes (staged: one 1,024-thread CTA per SM behind the TMA-staged track; unstaged: several
    256-thread CTAs per SM reading the track from global memory) and the host picks one by population size.  Forced each
    way on the same small population -- with a sensor offset, auto-reset and all 23 tracks -- both must be the oracle, bit
    for bit."""
    monkeypatch.setenv("OK_BEAM_KERNEL", kernel)
    names = ok.track_names()
    env, ora, tid = make_pair(names, 23 * 9, 32, movement_mode=mode, reward_mode=ok.REWARD_Q_PROGRESS, auto_reset=1, sensor_offset=2.5)
    assert env.launch_stats().block_threads == {"staged": 1024, "unstaged": 256}[kernel]
    pts = spread_points(ora, tid)
    env.reset(None, pts)
    ora.reset(None, pts)
    for step in range(150):
        env.launch_steps_random(step, 1)
        ora.fill_random_actions(step)
        ora.step()
        if step % 50 == 49:
            assert_same(env, ora, ctx=f"{kernel} kernel, step {step}")

"""GPU: ok_lidar_query -- lidar scans at arbitrary poses.  Bit for bit the agent path (ok_cast_rays on a population at the
same poses) in every ray-cast mode and beam-kernel shape, bit for bit the oracle (and the reference's own objects when
they are built) on hard poses, fans other than the env's, nullable outputs, no side effects, CUDA-graph capture."""
import numpy as np
import pytest
import torch

import openkitchen_b200 as ok
from openkitchen_b200 import _capi
from oracle.api import Oracle, have_ref
from tests.util import same_bits

pytestmark = pytest.mark.gpu

NAMES = ["obs", "hits", "hit_points", "hit_seg", "hit_t", "min_dist2", "crashed"]
C_NAMES = {"obs": "obs", "hits": "hit_rel", "hit_points": "hit_abs", "hit_seg": "hit_seg", "hit_t": "hit_t",
           "min_dist2": "min_dist2", "crashed": "crashed"}  # BatchEnv name -> agent buffer / OkLidarQuery field
MODES = {"beam": ok.RAYCAST_BEAM, "grid": ok.RAYCAST_GRID, "brute": ok.RAYCAST_BRUTE}


def _same(a, b):
    a = a.cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
    b = b.cpu().numpy() if torch.is_tensor(b) else np.asarray(b)
    return a.shape == b.shape and bool(same_bits(a, b).all())


def _mid_rollout(n, rays, **cfg):
    """a population over the 23 tracks after 60 random ticks with auto-reset, crash flags cleared, rays cast"""
    env = ok.BatchEnv(ok.track_names(), n, rays=rays, reward_mode=ok.REWARD_CMAES_PROGRESS, auto_reset=1, **cfg)
    env.step_random(60)
    env.crashed.zero_()
    env.cast_rays()
    return env


@pytest.mark.parametrize("offset", [0.0, 17.5])
@pytest.mark.parametrize("mode,shape", [("beam", "staged"), ("beam", "unstaged"), ("grid", None), ("brute", None)])
def test_equals_the_agent_path(monkeypatch, mode, shape, offset):
    if shape:
        monkeypatch.setenv("OK_BEAM_KERNEL", shape)
    n = 460 if mode == "brute" else 2300
    env = _mid_rollout(n, 32, raycast_mode=MODES[mode], sensor_offset=offset)
    got = env.lidar(env.pos_x, env.pos_y, env.rot, env.track_id.cuda())
    torch.cuda.synchronize()
    for nm in NAMES:
        assert _same(got[nm], env[C_NAMES[nm]]), nm
    assert env.env.launch_stats().block_threads == (256 if shape == "unstaged" else 1024)
    env.close()


def _hard_poses(env, rng, n, n_tracks):
    """poses on the lane, far outside the track window, exactly on boundary points, non-finite and huge coordinates,
    headings beyond +-10,000 degrees"""
    tid = rng.integers(0, n_tracks, n).astype(np.int32)
    x = rng.uniform(0.0, 1600.0, n).astype(np.float32)
    y = rng.uniform(0.0, 1400.0, n).astype(np.float32)
    rot = rng.uniform(-360.0, 360.0, n).astype(np.float32)
    for k in range(0, n, 3):
        cx, cy = env.track_array(int(tid[k]), "x"), env.track_array(int(tid[k]), "y")
        i = int(rng.integers(0, len(cx)))
        x[k], y[k] = cx[i] + np.float32(rng.normal(0, 4)), cy[i] + np.float32(rng.normal(0, 4))
    for k in range(1, n, 7):
        b = env.track_array(int(tid[k]), ("li", "lo", "ri", "ro")[k % 4])
        x[k], y[k] = b[int(rng.integers(0, len(b)))]
    x[2::11] += np.float32(3000.0)  # outside every table's window: uncovered cells, the grid walk from 0
    y[4::13] -= np.float32(2500.0)
    x[5], y[8], rot[11] = np.nan, np.nan, np.nan
    x[14], y[17], x[20], y[20] = np.float32(1e9), np.float32(-1e9), np.float32(-3e8), np.float32(7e8)
    rot[::5] += np.float32(10000.0) * np.sign(rng.standard_normal(len(rot[::5]))).astype(np.float32)
    rot[23], rot[26] = np.float32(123456.75), np.float32(-98765.5)
    return x, y, rot, tid


@pytest.mark.parametrize("rays", [5, 33])
@pytest.mark.parametrize("kind", ["port", "reference"])
def test_equals_the_oracle_on_hard_poses(kind, rays):
    if kind == "reference" and not have_ref():
        pytest.skip("oracle/_ref/libokref.so not built")
    names = ["Monza", "Spa", "Oschersleben", "Austin"]
    cfg = dict(sensor_range=137.5, sensor_offset=3.25)
    env = ok.Env(device=0, **cfg)
    for nm in names:
        env.add_named_track(nm)
    rng = np.random.default_rng(rays)
    n = 420
    x, y, rot, tid = _hard_poses(env, rng, n, len(names))
    fan = np.sort(rng.uniform(-100.0, 100.0, rays)).astype(np.float32)
    ora = Oracle(kind, **cfg)
    for nm in names:
        ora.add_track(ok.track_columns(nm))
    ora.alloc_agents(n, fan, tid)
    ora.buffer("pos_x")[:], ora.buffer("pos_y")[:], ora.buffer("rot")[:] = x, y, rot
    ora.buffer("crashed")[:] = 0
    ora.cast_rays()
    for mode in ("beam", "grid", "brute"):
        env.update_config(raycast_mode=MODES[mode])
        got = env.lidar_query(x, y, rot, tid, fan)
        for nm in NAMES:
            want = ora.buffer(C_NAMES[nm])
            assert got[nm].shape == want.shape, (mode, nm)
            bad = np.argwhere(~same_bits(got[nm], want))
            assert len(bad) == 0, (mode, nm, len(bad), tuple(bad[0]))
    env.close()


def test_fans_and_state():
    names = ["Monza", "Spa"]
    env = ok.BatchEnv(names, 512, rays=9, reward_mode=ok.REWARD_CMAES_PROGRESS, auto_reset=1)
    env.step_random(30)
    x, y, rot, tid = env.pos_x.clone(), env.pos_y.clone(), env.rot.clone(), env.track_id.cuda()
    other = (ok.ray_fan(7) * np.float32(0.5) + np.float32(3.0)).astype(np.float32)
    a = env.lidar(x, y, rot, tid, rays=other)
    # the agent path with that fan at those poses
    twin = ok.BatchEnv(names, 512, rays=other, reward_mode=ok.REWARD_CMAES_PROGRESS)
    twin.pos_x.copy_(x), twin.pos_y.copy_(y), twin.rot.copy_(rot)
    twin.cast_rays()
    # before any agent exists: an explicit fan is all it needs
    bare = ok.Env(device=0)
    for nm in names:
        bare.add_named_track(nm)
    c = bare.lidar_query(x.cpu().numpy(), y.cpu().numpy(), rot.cpu().numpy(), tid.cpu().numpy(), other)
    torch.cuda.synchronize()
    for nm in NAMES:
        assert _same(a[nm], twin[C_NAMES[nm]]), nm
        assert _same(a[nm], c[nm]), nm
    # a NULL fan is the env's own
    assert all(_same(env.lidar(x, y, rot, tid)[nm], env.lidar(x, y, rot, tid, rays=9)[nm]) for nm in NAMES)
    assert env.lidar(x, y, rot, tid)["obs"].shape == (512, 9)
    with pytest.raises(ok.OkError) as ex:
        bare.lidar_query(x.cpu().numpy(), y.cpu().numpy(), rot.cpu().numpy())
    assert ex.value.code == _capi.OK_ERR_STATE
    fan = torch.zeros(1025, device="cuda")
    for rays in (0, 1025):
        with pytest.raises(ok.OkError) as ex:
            env.env.lidar_query_device(x.data_ptr(), y.data_ptr(), rot.data_ptr(), 512, d_ray_deg=fan.data_ptr(), rays=rays,
                                       obs=torch.empty(512 * 1025, device="cuda").data_ptr())
        assert ex.value.code == _capi.OK_ERR_INVALID_ARG
    with pytest.raises(ok.OkError) as ex:
        env.env.lidar_query_device(None, y.data_ptr(), rot.data_ptr(), 512, rays=9)
    assert ex.value.code == _capi.OK_ERR_INVALID_ARG
    env.env.lidar_query_device(None, None, None, 0, rays=9)  # n == 0: nothing to do
    for e in (env, twin, bare):
        e.close()


def test_each_output_alone_equals_the_full_query():
    env = _mid_rollout(1150, 16)
    x, y, rot, tid = env.pos_x, env.pos_y, env.rot, env.track_id.cuda()
    full = env.lidar(x, y, rot, tid)
    for nm in NAMES:
        alone = env.lidar(x, y, rot, tid, outputs=[nm])
        assert list(alone) == [nm] and _same(alone[nm], full[nm]), nm
    env.close()


def test_no_side_effects():
    env = _mid_rollout(2300, 32)
    env.env.debug_stats(True)
    before = {nm: env[nm].clone() for nm in ok.BUFFERS}
    tiles, stats = env.env.debug_tiles(), env.env.launch_stats()
    x, y, rot, tid = env.pos_x.clone() + 1.5, env.pos_y.clone(), env.rot.clone() - 20.0, env.track_id.cuda()
    for _ in range(100):
        env.lidar(x, y, rot, tid)
    torch.cuda.synchronize()
    for nm in ok.BUFFERS:
        assert torch.equal(env[nm].view(torch.uint8), before[nm].view(torch.uint8)), nm
    assert np.array_equal(env.env.debug_tiles(), tiles)
    after = env.env.launch_stats()
    assert after.kernel_launches == stats.kernel_launches + 100
    assert (after.grid_blocks, after.tiles, after.block_threads, after.smem_bytes) == \
        (stats.grid_blocks, stats.tiles, stats.block_threads, stats.smem_bytes)
    assert env.env.debug_stats(False) == (0, 0, 0)
    env.close()


def test_capture():
    # an env that has never computed has no track arena yet: building it inside a capture is refused
    x = torch.rand(64, device="cuda") * 800.0
    y = torch.rand(64, device="cuda") * 600.0
    rot = torch.rand(64, device="cuda") * 360.0
    bare = ok.Env(device=0)
    bare.add_named_track("Monza")
    out = torch.empty(64 * 5, device="cuda")
    fan = torch.from_numpy(ok.ray_fan(5)).cuda()
    side = torch.cuda.Stream()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        out.add_(1.0)
        with pytest.raises(ok.OkError) as ex:
            bare.lidar_query_device(x.data_ptr(), y.data_ptr(), rot.data_ptr(), 64, d_ray_deg=fan.data_ptr(), rays=5, obs=out.data_ptr(),
                                    stream=torch.cuda.current_stream().cuda_stream)
    assert ex.value.code == _capi.OK_ERR_STATE and "outside the capture" in str(ex.value)
    # after one eager call the query is capturable and replays to the eager result
    env = _mid_rollout(1150, 32)
    px, py, prot, tid = env.pos_x.clone(), env.pos_y.clone(), env.rot.clone(), env.track_id.cuda()
    eager = env.lidar(px, py, prot, tid)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        captured = env.lidar(px, py, prot, tid)
    for t in captured.values():
        t.zero_()
    g.replay()
    torch.cuda.synchronize()
    for nm in NAMES:
        assert _same(captured[nm], eager[nm]), nm
    for e in (bare, env):
        e.close()


def test_no_index_leaves_its_array():
    """With a -DOK_CHECKED=1 library (tools/checked_build.sh) every table row, chunk, segment and pose index of the query
    kernel is range-checked; the beam-mode query over the hard poses must count zero violations."""
    names = ["Monza", "Spa", "Oschersleben", "Austin"]
    env = ok.Env(device=0, sensor_offset=3.25)
    for nm in names:
        env.add_named_track(nm)
    for rays in (5, 33):
        x, y, rot, tid = _hard_poses(env, np.random.default_rng(rays), 420, len(names))
        tid[::9] = 99  # clamped to the last track
        env.lidar_query(x, y, rot, tid, ok.ray_fan(rays))
    count, compiled_in = env.debug_violations()
    assert count == 0, f"{count} out-of-range indices"
    env.close()
    if not compiled_in:
        assert ok.LIB_PATH.endswith("libopenkitchen_b200.so")

"""GPU: ok_bev_query -- bird's-eye-view rasters at arbitrary poses.  Bit for bit the brute-force oracle (tests/bev_oracle.c) on all
23 tracks, on lane poses and hard poses, over image shapes, scales and forward shifts; one output above 2^31 bytes;
BatchEnv.bev's defaults; clamped track ids; no side effects; CUDA-graph capture; and a cross-check against the lidar,
which also pins the orientation of the image."""
import numpy as np
import pytest
import torch

import openkitchen_b200 as ok
from openkitchen_b200 import _capi
from tests.bev_oracle import BevOracle
from tests.test_gpu_lidar_query import _hard_poses

pytestmark = pytest.mark.gpu

MODES = {"beam": ok.RAYCAST_BEAM, "grid": ok.RAYCAST_GRID, "brute": ok.RAYCAST_BRUTE}
LOOPS = ("li", "lo", "ri", "ro")


@pytest.fixture(scope="module")
def world():
    """an env and the oracle with all 23 tracks"""
    env, ora = ok.Env(device=0), BevOracle()
    for nm in ok.track_names():
        env.add_named_track(nm)
        ora.add_track(ok.track_columns(nm))
    yield env, ora
    env.close()
    ora.close()


def _lane_poses(env, rng, per_track):
    """centre-line points with their headings, `per_track` on every track"""
    x, y, rot, tid = [], [], [], []
    for t in range(env.num_tracks()):
        cx, cy, hd = env.track_array(t, "x"), env.track_array(t, "y"), env.track_array(t, "heading")
        i = rng.integers(0, len(cx), per_track)
        x.append(cx[i]), y.append(cy[i]), rot.append(hd[i]), tid.append(np.full(per_track, t, np.int32))
    return tuple(np.concatenate(a) for a in (x, y, rot, tid))


def _poses(env, seed, lane_per_track, hard):
    rng = np.random.default_rng(seed)
    lx, ly, lr, lt = _lane_poses(env, rng, lane_per_track)
    hx, hy, hr, ht = _hard_poses(env, rng, hard, env.num_tracks())
    x, y, rot, tid = (np.concatenate(a) for a in ((lx, hx), (ly, hy), (lr, hr), (lt, ht)))
    rot[::4] = np.float32(-90.0)  # crops aligned with the window
    return x, y, rot, tid


def _oracle(ora, x, y, rot, tid, h, w, scale, ahead):
    return np.concatenate([ora.bev(int(tid[k]), x[k], y[k], rot[k], h, w, scale, ahead) for k in range(len(x))])


# every scale and forward shift on the small shapes; two of them on each of the larger ones (the oracle is brute force)
CASES = [((h, w), s, a) for (h, w) in ((1, 1), (1, 3)) for s in (0.25, 1.0, 3.5) for a in (0.0, 20.0)]
CASES += [((64, 64), 1.0, 0.0), ((64, 64), 3.5, 20.0), ((33, 97), 0.25, 20.0), ((33, 97), 1.0, 0.0),
          ((200, 7), 3.5, 0.0), ((200, 7), 0.25, 20.0)]


@pytest.mark.parametrize("shape,scale,ahead", CASES, ids=lambda v: str(v))
def test_equals_the_oracle(world, shape, scale, ahead):
    env, ora = world
    h, w = shape
    small = h * w <= 3
    x, y, rot, tid = _poses(env, h * 1000 + w, 12 if small else 1, 420 if small else 30)
    got = env.bev_query(x, y, rot, h, w, scale, ahead, track_id=tid)
    want = _oracle(ora, x, y, rot, tid, h, w, scale, ahead)
    assert got.shape == want.shape == (len(x), h, w)
    bad = np.argwhere(got != want)
    assert len(bad) == 0, (len(bad), tuple(bad[0]), int(got[tuple(bad[0])]), int(want[tuple(bad[0])]))
    if not small:
        assert set(np.unique(got)) == {ok.BEV_OFF, ok.BEV_WALL, ok.BEV_LANE}


def test_output_above_2gib(world):
    """70,000 poses x 256 x 128 = 2.29e9 bytes in one launch: every pixel index above 2^31 must land where it belongs"""
    env, ora = world
    n, h, w = 70_000, 256, 128
    rng = np.random.default_rng(7)
    x, y, rot, tid = _lane_poses(env, rng, (n + 22) // 23)
    x, y, rot, tid = x[:n], y[:n], rot[:n], tid[:n]
    rot = rot + rng.uniform(-30.0, 30.0, n).astype(np.float32)
    dev = [torch.from_numpy(a).cuda() for a in (x, y, rot, tid)]
    out = torch.empty((n, h, w), dtype=torch.uint8, device="cuda")
    env.bev_query_device(dev[0].data_ptr(), dev[1].data_ptr(), dev[2].data_ptr(), n, h, w, 0.5, out.data_ptr(), 10.0,
                         dev[3].data_ptr())
    sample = np.array([0, 1, 16383, 16384, 65535, 65536, n - 2, n - 1])  # pose 65,536 starts at byte 2^31
    got = out[torch.from_numpy(sample).cuda()].cpu().numpy()
    want = _oracle(ora, x[sample], y[sample], rot[sample], tid[sample], h, w, 0.5, 10.0)
    assert np.array_equal(got, want)
    del out


def test_unaligned_output_and_tails(world):
    """an output that starts off a 4-byte boundary and a total that is no multiple of 4: the byte-wise ends"""
    env, ora = world
    x, y, rot, tid = _poses(env, 11, 1, 30)
    dev = [torch.from_numpy(a).cuda() for a in (x, y, rot, tid)]
    n, h, w = len(x), 5, 7
    for off in range(4):
        buf = torch.full((n * h * w + 8,), 77, dtype=torch.uint8, device="cuda")
        env.bev_query_device(dev[0].data_ptr(), dev[1].data_ptr(), dev[2].data_ptr(), n, h, w, 2.0, buf.data_ptr() + off,
                             0.0, dev[3].data_ptr())
        b = buf.cpu().numpy()
        assert (b[:off] == 77).all() and (b[off + n * h * w:] == 77).all()
        assert np.array_equal(b[off:off + n * h * w].reshape(n, h, w), _oracle(ora, x, y, rot, tid, h, w, 2.0, 0.0))


def test_batch_env_defaults_and_ray_cast_modes():
    env = ok.BatchEnv(ok.track_names(), 2300, rays=8, reward_mode=ok.REWARD_CMAES_PROGRESS, auto_reset=1)
    env.step_random(40)
    a = env.bev(48, 40, 1.5, 8.0)
    b = env.bev(48, 40, 1.5, 8.0, x=env.pos_x.clone(), y=env.pos_y.clone(), rot=env.rot.clone(),
                track_id=env.track_id.clone())
    torch.cuda.synchronize()
    assert a.dtype == torch.uint8 and a.shape == (2300, 48, 40) and a.device.type == "cuda"
    assert torch.equal(a, b)
    assert torch.equal(env.bev()[:, 0, 0], env.bev(64, 64, 1.0, 0.0)[:, 0, 0])  # the defaults: 64 x 64, scale 1, ahead 0
    for mode in ("grid", "brute", "beam"):  # the raster does not depend on the ray-cast mode
        env.env.update_config(raycast_mode=MODES[mode])
        assert torch.equal(env.bev(48, 40, 1.5, 8.0), a), mode
    env.close()


def test_out_of_range_track_ids_are_clamped(world):
    env, _ = world
    x, y, rot, tid = _poses(env, 3, 2, 30)
    nt = env.num_tracks()
    wild = tid.copy()
    wild[::3], wild[1::3] = -5, nt + 40
    clamped = np.clip(wild, 0, nt - 1).astype(np.int32)
    assert np.array_equal(env.bev_query(x, y, rot, 16, 16, 2.0, track_id=wild),
                          env.bev_query(x, y, rot, 16, 16, 2.0, track_id=clamped))
    # no track id is track 0
    assert np.array_equal(env.bev_query(x, y, rot, 16, 16, 2.0), env.bev_query(x, y, rot, 16, 16, 2.0, track_id=np.zeros_like(tid)))


def test_before_alloc_agents_and_errors():
    bare = ok.Env(device=0)
    bare.add_named_track("Monza")
    ora = BevOracle()
    ora.add_track(ok.track_columns("Monza"))
    x, y, rot = bare.track_array(0, "x")[:20], bare.track_array(0, "y")[:20], bare.track_array(0, "heading")[:20]
    got = bare.bev_query(x, y, rot, 24, 24, 1.0)
    assert np.array_equal(got, _oracle(ora, x, y, rot, np.zeros(20, np.int32), 24, 24, 1.0, 0.0))
    assert (got[:, 11:13, 11:13] == ok.BEV_LANE).all()  # the pose itself sits on the lane
    q = _capi.OkBevQuery(n=0, height=8, width=8, scale=1.0)
    assert _capi.load().ok_bev_query(bare.h, q, None) == 0  # n == 0: nothing to do, NULL pointers allowed
    for bad in (dict(height=0), dict(width=1025), dict(scale=0.0), dict(scale=float("nan")), dict(ahead=float("inf"))):
        a = dict(x=x.ctypes.data, y=x.ctypes.data, rot=x.ctypes.data, n=1, height=8, width=8, scale=1.0, ahead=0.0,
                 out=got.ctypes.data)
        a.update(bad)
        assert _capi.load().ok_bev_query_host(bare.h, _capi.OkBevQuery(**a), None) == _capi.OK_ERR_INVALID_ARG, bad
    a = dict(x=x.ctypes.data, y=x.ctypes.data, rot=x.ctypes.data, n=1, height=8, width=8, scale=1.0, ahead=0.0, out=None)
    assert _capi.load().ok_bev_query_host(bare.h, _capi.OkBevQuery(**a), None) == _capi.OK_ERR_INVALID_ARG
    a.update(out=got.ctypes.data, n=-1)
    assert _capi.load().ok_bev_query_host(bare.h, _capi.OkBevQuery(**a), None) == _capi.OK_ERR_INVALID_ARG
    empty = ok.Env(device=0)
    a.update(n=1)
    assert _capi.load().ok_bev_query_host(empty.h, _capi.OkBevQuery(**a), None) == _capi.OK_ERR_STATE
    for e in (bare, empty):
        e.close()
    ora.close()


def test_no_side_effects():
    env = ok.BatchEnv(ok.track_names(), 2300, rays=32, reward_mode=ok.REWARD_CMAES_PROGRESS, auto_reset=1)
    env.step_random(60)
    env.cast_rays()
    env.env.debug_stats(True)
    before = {nm: env[nm].clone() for nm in ok.BUFFERS}
    tiles, stats = env.env.debug_tiles(), env.env.launch_stats()
    for _ in range(100):
        env.bev(64, 64, 1.0, 12.0)
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
    # an env that has never run the query has no band table yet: building it inside a capture is refused
    x = torch.rand(64, device="cuda") * 800.0
    y = torch.rand(64, device="cuda") * 600.0
    rot = torch.rand(64, device="cuda") * 360.0
    bare = ok.Env(device=0)
    bare.add_named_track("Monza")
    out = torch.empty((64, 16, 16), dtype=torch.uint8, device="cuda")
    side = torch.cuda.Stream()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=side):
        out.zero_()
        with pytest.raises(ok.OkError) as ex:
            bare.bev_query_device(x.data_ptr(), y.data_ptr(), rot.data_ptr(), 64, 16, 16, 1.0, out.data_ptr(),
                                  stream=torch.cuda.current_stream().cuda_stream)
    assert ex.value.code == _capi.OK_ERR_STATE and "outside the capture" in str(ex.value)
    # after one eager call the query is capturable and replays to the eager result
    env = ok.BatchEnv(ok.track_names(), 1150, rays=8, reward_mode=ok.REWARD_CMAES_PROGRESS, auto_reset=1)
    env.step_random(30)
    eager = env.bev(40, 56, 2.0, 5.0)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        captured = env.bev(40, 56, 2.0, 5.0)
    captured.zero_()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(captured, eager)
    for e in (bare, env):
        e.close()


def _near_edge(env, t, px, py, tol=1e-3):
    """float64: is (px, py) within tol px of an edge of one of the four loops of track t?"""
    q = np.array([px, py], dtype=np.float64)
    for nm in LOOPS:
        b = env.track_array(t, nm).astype(np.float64)
        a, d = np.roll(b, 1, axis=0), b - np.roll(b, 1, axis=0)
        s = np.clip(((q - a) * d).sum(1) / np.maximum((d * d).sum(1), 1e-300), 0.0, 1.0)
        if np.sqrt((((a + s[:, None] * d) - q) ** 2).sum(1)).min() < tol:
            return True
    return False


def test_agrees_with_the_lidar(world):
    """From a lane pose, the lidar's ray crosses no loop edge before its hit at t: the point halfway along it is LANE.  The
    1x1 image with ahead = t/2 at heading + ray angle samples that point; for the +90 / -90 degree rays so do column 2 /
    column 0 of a 1x3 image with scale = t/2 -- a mirrored image would put them on the wrong side."""
    env, _ = world
    env.update_config(sensor_offset=0.0)
    x, y, rot, tid = _lane_poses(env, np.random.default_rng(5), 6)
    fan = np.array([-90.0, 0.0, 90.0], dtype=np.float32)
    t = env.lidar_query(x, y, rot, tid, fan)["hit_t"]
    checked = 0
    for k in range(len(x)):
        pts = []
        for r in range(3):
            half = float(np.float32(t[k, r]) * np.float32(0.5))
            img = env.bev_query(x[k:k + 1], y[k:k + 1], (rot[k:k + 1] + fan[r]).astype(np.float32), 1, 1, 1.0, half,
                                track_id=tid[k:k + 1])
            pts.append((img[0, 0, 0], rot[k] + fan[r], half, 0.0))
        for r, col in ((2, 2), (0, 0)):
            half = float(np.float32(t[k, r]) * np.float32(0.5))
            img = env.bev_query(x[k:k + 1], y[k:k + 1], rot[k:k + 1], 1, 3, half, 0.0, track_id=tid[k:k + 1])
            pts.append((img[0, 0, col], rot[k] + fan[r], half, 0.0))
        for cls, ang, dist, _ in pts:
            checked += 1
            if cls != ok.BEV_LANE:
                a = np.deg2rad(np.float64(ang))
                px, py = x[k] + dist * np.cos(a), y[k] + dist * np.sin(a)
                assert _near_edge(env, int(tid[k]), px, py), (k, int(cls), float(ang), dist)
    assert checked == 5 * len(x)


def test_no_index_leaves_its_array(world):
    """With a -DOK_CHECKED=1 library (tools/checked_build.sh) every band, list and pose index of the query kernel is
    range-checked; the hard poses must count zero violations."""
    env, _ = world
    x, y, rot, tid = _poses(env, 9, 2, 420)
    tid[::9] = 99  # clamped to the last track
    for h, w, s, a in ((1, 1, 1.0, 0.0), (33, 97, 3.5, 20.0), (200, 7, 0.25, 0.0)):
        env.bev_query(x, y, rot, h, w, s, a, track_id=tid)
    count, compiled_in = env.debug_violations()
    assert count == 0, f"{count} out-of-range indices"
    if not compiled_in:
        assert ok.LIB_PATH.endswith("libopenkitchen_b200.so")

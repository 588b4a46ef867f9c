"""GPU: the *_host entry points of one env share its staging buffer.  Interleaved on one env -- track, lidar and
bird's-eye-view queries, resets and sincosf -- at sizes that grow the buffer, reuse it for smaller calls and grow it
again, every host-form result is bit for bit the device-pointer form on the same inputs, and a host-array reset leaves
the state a device-array reset leaves on a twin env."""
import ctypes as C

import numpy as np
import pytest
import torch

import openkitchen_b200 as ok
from openkitchen_b200 import _capi
from openkitchen_b200.env import LIDAR_OUTPUTS
from tests.util import same_bits

pytestmark = pytest.mark.gpu

NAMES = ["Monza", "Spa", "Oschersleben", "Austin"]
AGENTS, RAYS = 2048, 9


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _same(host, dev):
    return bool(same_bits(host, dev.cpu().numpy().reshape(host.shape)).all())


def _poses(env, rng, n):
    """poses near the centre lines of the four tracks"""
    tid = rng.integers(0, len(NAMES), n).astype(np.int32)
    x, y = np.empty(n, np.float32), np.empty(n, np.float32)
    for t in range(len(NAMES)):
        k = np.flatnonzero(tid == t)
        cx, cy = env.track_array(t, "x"), env.track_array(t, "y")
        i = rng.integers(0, len(cx), len(k))
        x[k] = cx[i] + rng.normal(0, 5, len(k)).astype(np.float32)
        y[k] = cy[i] + rng.normal(0, 5, len(k)).astype(np.float32)
    return x, y, rng.uniform(-360.0, 360.0, n).astype(np.float32), tid


def _check_track_query(env, x, y, tid):
    got = env.track_query(x, y, tid)
    n = len(x)
    want = (torch.empty(n, dtype=torch.int32, device="cuda"), torch.empty(n, device="cuda"), torch.empty(n, device="cuda"))
    d = [_dev(a) for a in (x, y, tid)]  # held until the query has run: a freed tensor's block is handed out again
    env.track_query_device(*(a.data_ptr() for a in d), n, *(w.data_ptr() for w in want))
    torch.cuda.synchronize()
    for name, g, w in zip(("nearest_idx", "dist_lane_center", "dist_boundary"), got, want):
        assert _same(g, w), ("track_query", name)


def _check_lidar(env, x, y, rot, tid, fan, outputs):
    """ok_lidar_query_host against ok_lidar_query with the outputs named (BatchEnv names) and every other one NULL"""
    n, rays = len(x), (env.rays if fan is None else len(fan))
    host = {nm: np.empty(LIDAR_OUTPUTS[nm][2](n, rays), dtype=LIDAR_OUTPUTS[nm][1]) for nm in outputs}
    q = _capi.OkLidarQuery(x=x.ctypes.data, y=y.ctypes.data, rot=rot.ctypes.data, track_id=tid.ctypes.data, n=n,
                           ray_deg=None if fan is None else fan.ctypes.data, rays=rays,
                           **{LIDAR_OUTPUTS[nm][0]: a.ctypes.data for nm, a in host.items()})
    _capi.check(env.lib.ok_lidar_query_host(env.h, C.byref(q), None))
    dev = {nm: torch.from_numpy(np.empty_like(a)).cuda() for nm, a in host.items()}
    d_in = [_dev(a) for a in (x, y, rot, tid)]
    d_fan = None if fan is None else _dev(fan)
    env.lidar_query_device(*(a.data_ptr() for a in d_in[:3]), n, d_in[3].data_ptr(),
                           None if d_fan is None else d_fan.data_ptr(), rays,
                           **{LIDAR_OUTPUTS[nm][0]: t.data_ptr() for nm, t in dev.items()})
    torch.cuda.synchronize()
    for nm in outputs:
        assert _same(host[nm], dev[nm]), ("lidar", nm, fan is None)


def _check_bev(env, x, y, rot, tid):
    h, w, scale, ahead = 40, 56, 1.5, 12.0
    got = env.bev_query(x, y, rot, h, w, scale, ahead, track_id=tid)
    want = torch.empty((len(x), h, w), dtype=torch.uint8, device="cuda")
    d = [_dev(a) for a in (x, y, rot, tid)]
    env.bev_query_device(d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), len(x), h, w, scale, want.data_ptr(), ahead,
                         d[3].data_ptr())
    torch.cuda.synchronize()
    assert _same(got, want), "bev"


def _reset_pair(env, twin, rng, n, given, step):
    """the same reset on both envs, env through host arrays and twin through device arrays, then one tick of each"""
    tid = np.arange(AGENTS) * len(NAMES) // AGENTS
    npts = np.array([env.track_info(t).n_points for t in range(len(NAMES))])
    idx = rng.permutation(AGENTS)[:n].astype(np.int64) if given else None
    agents = idx if given else np.arange(n)
    pts = (rng.integers(0, 1 << 20, n) % npts[tid[agents]]).astype(np.int32)
    alpha = rng.uniform(0.0, 1.0, n).astype(np.float32) if given else None
    hoff = rng.uniform(-15.0, 15.0, n).astype(np.float32) if given else None
    env.reset(idx, pts, alpha, hoff)
    d = [None if a is None else _dev(a) for a in (idx, pts, alpha, hoff)]
    twin.reset_device(*(None if t is None else t.data_ptr() for t in d), n)
    torch.cuda.synchronize()
    for e in (env, twin):
        e.launch_steps_random(step, 1)
    for nm in ok.BUFFERS:
        assert same_bits(env.read(nm), twin.read(nm)).all(), ("reset", nm, n, given)


def test_entry_points_share_one_stage():
    rng = np.random.default_rng(11)
    tid = (np.arange(AGENTS) * len(NAMES) // AGENTS).astype(np.int32)
    env, twin = ok.Env(device=0), ok.Env(device=0)
    for e in (env, twin):
        for nm in NAMES:
            e.add_named_track(nm)
        e.alloc_agents(AGENTS, ok.ray_fan(RAYS), tid)
    fresh = ok.Env(device=0)  # sincosf on an env whose stage no other call has used
    fan = np.sort(rng.uniform(-120.0, 120.0, 33)).astype(np.float32)
    step = 0
    for n in (3000, 37, 5000):  # grown, reused by smaller calls, grown again
        x, y, rot, qt = _poses(env, rng, n)
        _check_track_query(env, x, y, qt)
        _check_lidar(env, x, y, rot, qt, fan, list(LIDAR_OUTPUTS))
        _reset_pair(env, twin, rng, min(n, AGENTS), True, step)
        _check_lidar(env, x, y, rot, qt, None, list(LIDAR_OUTPUTS))
        _check_bev(env, x, y, rot, qt)
        _check_lidar(env, x, y, rot, qt, fan, ["hit_seg", "crashed"])
        _reset_pair(env, twin, rng, min(n, AGENTS), False, step + 1)
        s = rng.uniform(-1e4, 1e4, 64 * n).astype(np.float32)
        got, want = env.eval_sincosf(s), fresh.eval_sincosf(s)
        assert all(same_bits(g, w).all() for g, w in zip(got, want)), "sincosf"
        step += 2
    for e in (env, twin, fresh):
        e.close()

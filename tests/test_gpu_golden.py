"""GPU: the CUDA path against the committed golden vectors (tests/golden/traces.npz, minted from the
reference's own objects by tools/make_golden.py, and traces_live.npz, the live comparisons' scenarios) -- no oracle in
the loop, bit-exact."""
import os
import sys

import numpy as np
import pytest

import openkitchen_b200 as ok
from tests.util import same_bits

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "..", "tools"))
import make_golden as mg  # noqa: E402

pytestmark = pytest.mark.gpu
GOLD = np.load(os.path.join(os.path.dirname(__file__), "golden", "traces.npz"))
LIVE_GOLD = np.load(os.path.join(os.path.dirname(__file__), "golden", "traces_live.npz"))


@pytest.mark.parametrize("raycast", [ok.RAYCAST_BEAM, ok.RAYCAST_GRID, ok.RAYCAST_BRUTE])
@pytest.mark.parametrize("name", list(mg.SCENARIOS))
def test_cuda_path_matches_golden(name, raycast):
    tracks, n, rays, cfg, ticks, cps = mg.SCENARIOS[name]
    if raycast == ok.RAYCAST_BRUTE and ticks > 400:
        ticks, cps = 101, [c for c in cps if c <= 100]
    tracks = tracks or ok.track_names()
    env = ok.Env(device=0, raycast_mode=raycast, **cfg)
    pts_per = []
    for t in tracks:
        env.add_named_track(t)
        pts_per.append(len(ok.track_columns(t)[0]))
    tid = (np.arange(n) * len(tracks) // n).astype(np.int32)
    env.alloc_agents(n, mg.fan_of(rays), tid)
    pts = np.array([(i * 2654435761 % 2**32) % pts_per[int(tid[i])] for i in range(n)], dtype=np.int32)
    env.reset(None, pts)
    checked = 0
    for s in range(ticks):
        env.launch_steps_random(s, 1)
        if s in cps:
            for b in ok.BUFFERS:
                got, want = env.read(b), GOLD[f"{name}/{s}/{b}"]
                bad = ~same_bits(got, want)
                assert not bad.any(), f"{name} tick {s} buffer {b}: {int(bad.sum())} mismatches"
                checked += 1
    assert checked == len(cps) * len(ok.BUFFERS)


@pytest.mark.parametrize("raycast", [ok.RAYCAST_BEAM, ok.RAYCAST_GRID, ok.RAYCAST_BRUTE])
@pytest.mark.parametrize("name", list(mg.LIVE_SCENARIOS))
def test_cuda_path_matches_live_golden(name, raycast):
    """tests/golden/traces_live.npz: drawn reset points, lane and heading offsets, reward modes 1-7, sensor offsets and
    a non-default crash threshold"""
    tracks, n, fan, cfg, ticks, cps, tid, idx, pts, alpha, hoff = mg.live_inputs(name)
    cps = mg.golden_checkpoints(name)
    env = ok.Env(device=0, raycast_mode=raycast, **cfg)
    for t in tracks:
        env.add_named_track(t)
    env.alloc_agents(n, fan, tid)
    env.reset(idx, pts, alpha, hoff)
    checked = 0
    for s in range(cps[-1] + 1):
        env.launch_steps_random(s, 1)
        if s in cps:
            for b in ok.BUFFERS:
                got, want = env.read(b), LIVE_GOLD[f"{name}/{s}/{b}"]
                bad = ~same_bits(got, want)
                assert not bad.any(), f"{name} tick {s} buffer {b}: {int(bad.sum())} mismatches"
                checked += 1
    env.close()
    assert checked == len(cps) * len(ok.BUFFERS)

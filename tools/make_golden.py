#!/usr/bin/env python
"""Mint the golden vectors under tests/golden/ from the REFERENCE ITSELF run here:
oracle/_ref/libokref.so = the unmodified reference Agent.cpp + RaceTrack.cpp driven by
oracle/ref_harness.cpp (see oracle/Makefile).  The reference ships no tests or fixtures of its own
(SURVEY.md section 4), so these are the pins for the oracle and, through it, for the CUDA path.

    OPENKITCHEN_REF=<checkout> make -C oracle && python tools/make_golden.py            # all three files
    python tools/make_golden.py --live-from-port                                       # traces_live.npz only

Contents
  tracks.npz        per track: CRC32 of every RaceTrack / TrackSegments array + first/last rows
  traces.npz        per scenario: full state + lidar buffers at a few checkpoints of a scripted rollout
  traces_live.npz   the same for LIVE_SCENARIOS: the reset draws, reward modes, sensor offsets and crash threshold of
                    the live comparisons in tests/test_oracle_golden.py

`--live-from-port` mints traces_live.npz from the C restatement (oracle/ok_oracle.c) instead of the reference's objects.
It gives the same bits only while the restatement is unchanged since the live comparisons last passed against those
objects on exactly these scenarios.  The committed traces_live.npz was minted that way from oracle/ok_oracle.c as of
commit 07333d5, the version the live comparisons were run against the reference's objects with (the sensor-offset one
was added after it, in 2d0850c); the file has not changed since.
"""
import os
import sys
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import openkitchen_b200 as ok  # noqa: E402  (track pack + ray fan helpers only)
from oracle.api import BUF, Oracle  # noqa: E402

TRACK_ARRAYS = ["x", "y", "w_right", "w_left", "heading", "li", "lo", "ri", "ro", "segments"]

# name: (tracks, n_agents, rays/fan, config, ticks, checkpoints)
SCENARIOS = {
    # BASELINE config 0: one agent on Monza, Q-learning fan, VELOCITY mode
    "c1_single_monza": (["Monza"], 1, [-70, -30, 0, 30, 70], dict(movement_mode=0, reward_mode=1, auto_reset=1), 1000,
                        [0, 1, 10, 100, 500, 999]),
    # BASELINE config 1 shape (reduced population): Silverstone, 32 rays, ACCELERATION mode
    "c2_silverstone_accel": (["Silverstone"], 64, 32, dict(movement_mode=1, reward_mode=6, auto_reset=0), 400,
                             [0, 50, 200, 201, 399]),
    # BASELINE config 2 shape (reduced population): all 23 tracks, 32 rays, random actions, auto-reset
    "c3_all_tracks": (None, 92, 32, dict(movement_mode=0, reward_mode=2, auto_reset=1), 300, [0, 20, 100, 299]),
    # default 15-ray fan, lane-centre reward, no auto reset (agents crash and keep stale hits)
    "default_fan_lane_center": (["Spa", "Austin"], 40, 15, dict(movement_mode=0, reward_mode=7, auto_reset=0), 250,
                                [0, 30, 249]),
}


# The live comparisons of tests/test_oracle_golden.py (restatement vs the reference's objects), as scenarios.
# name: (tracks, n_agents, rays, config, ticks, checkpoints, seed of the reset draws, whether the lane offset and heading
# offset are drawn too).  Agents are dealt round-robin over the tracks.
LIVE_SCENARIOS = {}
for _mode, _reward in [(0, 1), (0, 2), (1, 7), (1, 5), (0, 4), (0, 3), (1, 6)]:
    LIVE_SCENARIOS[f"live_m{_mode}_r{_reward}"] = (
        ["Monza", "Zandvoort", "Spa"], 60, 15, dict(movement_mode=_mode, reward_mode=_reward, auto_reset=1), 150,
        [s for s in range(150) if s % 25 == 0 or s == 149], 7, True)
for _mode in (0, 1):
    for _offset in (3.0, -5.0):
        _ticks = 120 if _mode == 0 else 400  # the acceleration mode's action set builds speed slowly
        LIVE_SCENARIOS[f"offset_m{_mode}_{_offset:+g}"] = (
            ["Monza", "Sepang"], 48, 9, dict(movement_mode=_mode, reward_mode=1, auto_reset=1, sensor_offset=_offset,
                                             collision_dist2=3.5), _ticks,
            [s for s in range(_ticks) if s % 20 == 0 or s == _ticks - 1], 11, False)


def live_inputs(name):
    """(tracks, n, fan, config, ticks, checkpoints, track ids, agent ids, reset points, lane offsets, heading offsets)"""
    tracks, n, rays, cfg, ticks, cps, seed, offsets = LIVE_SCENARIOS[name]
    tid = (np.arange(n) % len(tracks)).astype(np.int32)
    pts_per = [len(ok.track_columns(t)[0]) for t in tracks]
    rng = np.random.default_rng(seed)
    idx = np.arange(n, dtype=np.int64)
    pts = np.array([rng.integers(0, pts_per[t]) for t in tid], dtype=np.int32)
    alpha = hoff = None
    if offsets:
        alpha = (rng.integers(10, 91, size=n) / np.float32(100)).astype(np.float32)
        hoff = rng.integers(-90, 91, size=n).astype(np.float32)
    return tracks, n, fan_of(rays), cfg, ticks, cps, tid, idx, pts, alpha, hoff


def golden_checkpoints(name):
    """the checkpoints traces_live.npz keeps (three per scenario, to stay under 1 MB): the second, the middle, the last"""
    cps = LIVE_SCENARIOS[name][5]
    return [cps[1], cps[len(cps) // 2], cps[-1]]


def run_live_scenario(kind, name, checkpoints=None):
    """LIVE_SCENARIOS[name] through the oracle `kind`: {"name/tick/buffer": array} at every checkpoint (or at
    `checkpoints`), and "name/crashed_seen": whether any agent crashed on any tick"""
    tracks, n, fan, cfg, ticks, cps, tid, idx, pts, alpha, hoff = live_inputs(name)
    cps = cps if checkpoints is None else checkpoints
    o = Oracle(kind, **cfg)
    for t in tracks:
        o.add_track(ok.track_columns(t))
    o.alloc_agents(n, fan, tid)
    o.reset(idx, pts, alpha, hoff)
    out, crashed_seen = {}, False
    for s in range(ticks):
        o.fill_random_actions(s)
        o.step()
        crashed_seen = crashed_seen or bool(o.buffer("crashed").any())
        if s in cps:
            for b in BUF:
                out[f"{name}/{s}/{b}"] = o.buffer(b).copy()
    out[f"{name}/crashed_seen"] = np.array([crashed_seen])
    o.close()
    return out


def fan_of(spec):
    return ok.ray_fan(spec) if np.isscalar(spec) else np.asarray(spec, dtype=np.float32)


def run_scenario(kind, name):
    tracks, n, rays, cfg, ticks, cps = SCENARIOS[name]
    tracks = tracks or ok.track_names()
    o = Oracle(kind, **cfg)
    for t in tracks:
        o.add_track(ok.track_columns(t))
    tid = (np.arange(n) * len(tracks) // n).astype(np.int32)
    o.alloc_agents(n, fan_of(rays), tid)
    pts = np.array([(i * 2654435761 % 2**32) % o.track_points(int(tid[i])) for i in range(n)], dtype=np.int32)
    o.reset(None, pts)
    out = {}
    for s in range(ticks):
        o.fill_random_actions(s)
        o.step()
        if s in cps:
            for b in BUF:
                out[f"{name}/{s}/{b}"] = o.buffer(b).copy()
    return out


def save(name, arrays):
    path = os.path.join(ROOT, "tests", "golden", name)
    np.savez_compressed(path, **arrays)
    print(name, os.path.getsize(path), "bytes")


def main():
    live = {}
    if "--live-from-port" in sys.argv[1:]:
        for name in LIVE_SCENARIOS:
            live.update(run_live_scenario("port", name, golden_checkpoints(name)))
        save("traces_live.npz", live)
        return
    ref = Oracle("reference")
    tr = {}
    for nm in ok.track_names():
        t = ref.add_track(ok.track_columns(nm))
        for a in TRACK_ARRAYS:
            arr = ref.track_array(t, a)
            tr[f"{nm}/{a}/crc"] = np.array([zlib.crc32(arr.tobytes())], dtype=np.uint32)
            tr[f"{nm}/{a}/shape"] = np.array(arr.shape, dtype=np.int32)
            tr[f"{nm}/{a}/head"] = arr.reshape(arr.shape[0], -1)[:2].copy()
            tr[f"{nm}/{a}/tail"] = arr.reshape(arr.shape[0], -1)[-2:].copy()
    save("tracks.npz", tr)
    traces = {}
    for name in SCENARIOS:
        traces.update(run_scenario("reference", name))
    save("traces.npz", traces)
    for name in LIVE_SCENARIOS:
        live.update(run_live_scenario("reference", name, golden_checkpoints(name)))
    save("traces_live.npz", live)


if __name__ == "__main__":
    main()

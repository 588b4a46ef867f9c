"""CPU: the plain-C oracle (oracle/ok_oracle.c) against the golden vectors minted from the reference's
own objects (tools/make_golden.py -> tests/golden/), and -- when oracle/_ref is built -- against
those objects live.  Bit-exact on every buffer.  traces_live.npz stores the result of the live comparisons' scenarios
(see tools/make_golden.py for how it was minted), so that they are checked where the reference is absent too."""
import os
import sys
import zlib

import numpy as np
import pytest

import openkitchen_b200 as ok
from oracle.api import BUF, Oracle, have_ref
from tests.util import same_bits

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "..", "tools"))
import make_golden as mg  # noqa: E402

GOLD = os.path.join(os.path.dirname(__file__), "golden")
# a checkout of the original project (not part of this repository): its track CSVs, when present
REF = os.environ.get("OPENKITCHEN_REF")
REF_TRACKS = os.path.join(REF, "tracks") if REF else None


@pytest.fixture(scope="module")
def tracks_gold():
    return np.load(os.path.join(GOLD, "tracks.npz"))


@pytest.fixture(scope="module")
def traces_gold():
    return np.load(os.path.join(GOLD, "traces.npz"))


def test_oracle_tracks_match_golden(tracks_gold):
    o = Oracle("port")
    for nm in ok.track_names():
        t = o.add_track(ok.track_columns(nm))
        for a in mg.TRACK_ARRAYS:
            arr = o.track_array(t, a)
            assert tuple(tracks_gold[f"{nm}/{a}/shape"]) == arr.shape
            assert zlib.crc32(arr.tobytes()) == int(tracks_gold[f"{nm}/{a}/crc"][0]), (nm, a)
            assert same_bits(arr.reshape(arr.shape[0], -1)[:2], tracks_gold[f"{nm}/{a}/head"]).all()
            assert same_bits(arr.reshape(arr.shape[0], -1)[-2:], tracks_gold[f"{nm}/{a}/tail"]).all()
    assert o.track_segments(ok.track_names().index("Monza")) == 4636  # SURVEY.md 8: 4(P-1)+4
    assert sum(o.track_segments(i) for i in range(23)) == 90676


@pytest.mark.parametrize("name", list(mg.SCENARIOS))
def test_oracle_traces_match_golden(name, traces_gold):
    got = mg.run_scenario("port", name)
    assert got, "scenario produced no checkpoints"
    for key, arr in got.items():
        assert same_bits(arr, traces_gold[key]).all(), key


@pytest.fixture(scope="module")
def live_gold():
    return np.load(os.path.join(GOLD, "traces_live.npz"))


@pytest.mark.parametrize("name", list(mg.LIVE_SCENARIOS))
def test_oracle_live_scenarios_match_golden(name, live_gold):
    """the live comparisons below, against their stored result (tests/golden/traces_live.npz): every buffer, bit-exact"""
    cps = mg.golden_checkpoints(name)
    got = mg.run_live_scenario("port", name, cps)
    assert len(got) == len(cps) * len(BUF) + 1
    for key, arr in got.items():
        assert same_bits(arr, live_gold[key]).all(), key
    if name.startswith("offset"):
        assert got[f"{name}/crashed_seen"][0], "nobody crashed: the changed threshold was never exercised"


def _live_pair(name):
    """LIVE_SCENARIOS[name] through the restatement and through the reference's objects: every buffer at every
    checkpoint, bit-exact"""
    a, b = mg.run_live_scenario("port", name), mg.run_live_scenario("reference", name)
    assert a.keys() == b.keys()
    for key in a:
        assert same_bits(a[key], b[key]).all(), key
    return a


@pytest.mark.skipif(not have_ref(), reason="oracle/_ref not built (needs the original project's sources: OPENKITCHEN_REF)")
@pytest.mark.parametrize("mode,reward", [(0, 1), (0, 2), (1, 7), (1, 5), (0, 4), (0, 3), (1, 6)])
def test_oracle_vs_reference_objects_live(mode, reward):
    _live_pair(f"live_m{mode}_r{reward}")  # Monza, Zandvoort, Spa; 60 agents, drawn reset points and offsets


def test_track_csv_writer_round_trips_the_pack(tmp_path):
    """write_track_csv re-emits every packed track so that strtof reads back the very same columns"""
    o = Oracle("port")
    for nm in ok.track_names():
        t_pack = o.add_track(ok.track_columns(nm))
        p = tmp_path / f"{nm}.csv"
        ok.write_track_csv(nm, str(p))
        t_rt = o.load_track_csv(str(p))
        for a in ("x", "y", "w_right", "w_left", "segments"):
            assert same_bits(o.track_array(t_pack, a), o.track_array(t_rt, a)).all(), (nm, a)


@pytest.mark.skipif(not (REF_TRACKS and os.path.isdir(REF_TRACKS)), reason="the original project's track CSVs are not present (OPENKITCHEN_REF)")
def test_track_pack_matches_reference_csvs(tmp_path):
    """the packed columns are exactly what strtof parses out of the reference's CSV files, and the
    CSV writer round-trips them"""
    o = Oracle("port")
    for nm in ok.track_names():
        t_csv = o.load_track_csv(os.path.join(REF_TRACKS, f"{nm}.csv"))
        t_pack = o.add_track(ok.track_columns(nm))
        p = tmp_path / f"{nm}.csv"
        ok.write_track_csv(nm, str(p))
        t_rt = o.load_track_csv(str(p))
        for a in ("x", "y", "w_right", "w_left", "segments"):
            ref = o.track_array(t_csv, a)
            assert same_bits(ref, o.track_array(t_pack, a)).all(), (nm, a)
            assert same_bits(ref, o.track_array(t_rt, a)).all(), (nm, a)


@pytest.mark.skipif(not have_ref(), reason="oracle/_ref not built (needs the original project's sources: OPENKITCHEN_REF)")
@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("offset", [3.0, -5.0])
def test_oracle_vs_reference_objects_with_a_sensor_offset(mode, offset):
    """Agent::sensor_offset_ (Agent.h:69, CollisionChecker.cu:122-126: the lidar origin is shifted along the heading) and the
    crash threshold of CollisionChecker.cu:167 -- what the reference's objects let one vary (dt, speed limit, sensor range
    and the standstill window are compile-time constants there: Agent.h:10-12, Environment.h:19-20) -- in the C restatement
    against the reference's own objects.  The GPU tests compare the CUDA path with the restatement on the same settings
    (tests/test_gpu_parity_gaps.py): this closes the chain CUDA == restatement == reference for them."""
    name = f"offset_m{mode}_{offset:+g}"
    assert _live_pair(name)[f"{name}/crashed_seen"][0], "nobody crashed: the changed threshold was never exercised"

"""CPU: the C-ABI library loads, exports every symbol include/openkitchen_b200.h declares, builds tracks
bit-identically to the reference on the host, and refuses loudly to compute without a GPU."""
import ctypes as C
import os
import re
import sys
import zlib

import numpy as np
import pytest

import openkitchen_b200 as ok
from openkitchen_b200 import _capi
from tests.util import same_bits

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


def test_library_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "openkitchen_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(ok_[a-z_0-9]+)\s*\(", header))
    assert len(declared) >= 25
    lib = C.CDLL(_capi.LIB_PATH)
    missing = [n for n in sorted(declared) if not hasattr(lib, n)]
    assert not missing, f"library does not export: {missing}"
    assert declared == set(_capi.SIGNATURES), "ctypes table and header disagree"
    assert _capi.load().ok_abi_version() == 2


def test_capi_allocates_device_memory_in_one_place():
    """Pool, don't free (DESIGN.md §7): in ok_capi.cu, cudaMalloc and cudaFree are called only by dev_alloc and CudaFree,
    the owners every buffer goes through, and by the measurement-only ok_pcie_probe.  The *_host entry points stage
    through the env's pooled buffer.  One predicate answers "is this stream capturing?"."""
    src = open(os.path.join(ROOT, "openkitchen_b200", "csrc", "ok_capi.cu")).read()
    src = re.sub(r"//[^\n]*", "", src)
    callers = {"cudaMalloc": set(), "cudaFree": set()}
    owner = None
    for line in src.splitlines():
        # a definition at column 0 names the function or struct the lines below belong to
        m = re.match(r"(?:template\s*<[^>]*>\s*)?(?:struct\s+(\w+)|[A-Za-z_][^(;=]*?\b(\w+)\s*\()", line)
        if m and not line.startswith(("extern", "namespace")):
            owner = m.group(1) or m.group(2)
        for fn in callers:
            if re.search(rf"\b{fn}\s*\(", line):
                callers[fn].add(owner)
    assert callers == {"cudaMalloc": {"dev_alloc", "ok_pcie_probe"}, "cudaFree": {"CudaFree", "ok_pcie_probe"}}, callers
    assert len(re.findall(r"\bcudaStreamIsCapturing\s*\(", src)) == 1


def test_config_defaults_are_the_reference_constants():
    c = _capi.OkConfig()
    _capi.load().ok_config_default(C.byref(c))
    assert (c.sensor_range, c.speed_limit, c.collision_dist2) == (200.0, 100.0, 2.0)  # Agent.h:10-11, CollisionChecker.cu:167
    assert c.dt == np.float32(0.016) and c.standstill_period == 200 and c.standstill_threshold == 20.0
    assert c.movement_mode == ok.MOVE_VELOCITY and c.sensor_offset == 0.0 and c.auto_reset == 0


def test_no_gpu_means_no_compute():
    """host-only env: tracks work, every compute entry point fails with OK_ERR_NO_DEVICE"""
    with ok.Env(device=-1) as e:
        e.add_named_track("Monza")
        with pytest.raises(ok.OkError) as ex:
            e.alloc_agents(4, ok.ray_fan(5))
        assert ex.value.code == _capi.OK_ERR_NO_DEVICE
        for call in (e.cast_rays, e.launch_step, lambda: e.launch_steps_random(0, 1)):
            with pytest.raises(ok.OkError) as ex:
                call()
            assert ex.value.code == _capi.OK_ERR_NO_DEVICE


def test_host_track_builder_matches_golden():
    gold = np.load(os.path.join(GOLD, "tracks.npz"))
    with ok.Env(device=-1) as e:
        for nm in ok.track_names():
            t = e.add_named_track(nm)
            for a in ("x", "y", "w_right", "w_left", "heading", "li", "lo", "ri", "ro", "segments"):
                arr = e.track_array(t, a)
                assert zlib.crc32(arr.tobytes()) == int(gold[f"{nm}/{a}/crc"][0]), (nm, a)
            info = e.track_info(t)
            assert info.n_segments == 4 * (info.n_points - 1) + 4
            assert 0 < info.blob_bytes <= 226 * 1024 and info.grid_items >= info.n_segments


def test_csv_loader_and_error_paths(tmp_path):
    with ok.Env(device=-1) as e:
        p = tmp_path / "Monza.csv"
        ok.write_track_csv("Monza", str(p))
        a = e.load_track_csv(str(p))
        b = e.add_named_track("Monza")
        assert same_bits(e.track_array(a, "segments"), e.track_array(b, "segments")).all()
        with pytest.raises(ok.OkError) as ex:
            e.load_track_csv(str(tmp_path / "missing.csv"))
        assert ex.value.code == _capi.OK_ERR_IO
        bad = tmp_path / "bad.csv"
        bad.write_text("# x_m,y_m,w_tr_right_m,w_tr_left_m\n1.0,2.0,3.0\n")
        with pytest.raises(ok.OkError):
            e.load_track_csv(str(bad))
        with pytest.raises(ok.OkError) as ex:
            e.add_track((np.zeros(1), np.zeros(1), np.ones(1), np.ones(1)))
        assert ex.value.code == _capi.OK_ERR_INVALID_ARG
    with pytest.raises(ok.OkError):
        ok.Env(device=-1, movement_mode=2)  # MANUAL is not supported
    with pytest.raises(ok.OkError):
        ok.Env(device=-1, grid_cell=0.1)


def test_grid_registers_every_segment_with_margin():
    """every segment appears in every cell its 1/16 px neighbourhood touches (sampled along its length)"""
    lib = _capi.load()
    with ok.Env(device=-1) as e:
        t = e.add_named_track("Spa")
        info = e.track_info(t)
        seg = e.track_array(t, "segments")
        assert info.grid_cell == 8.0
        # sample points along each segment must fall inside the clip box (ring of empty cells around it)
        x0, y0, c = info.grid_x0, info.grid_y0, info.grid_cell
        for s in seg[:: max(1, len(seg) // 400)]:
            for u in np.linspace(0, 1, 5):
                px, py = s[0] + u * (s[2] - s[0]), s[1] + u * (s[3] - s[1])
                ix, iy = int((px - x0) // c), int((py - y0) // c)
                assert 1 <= ix <= info.grid_nx - 2 and 1 <= iy <= info.grid_ny - 2


def test_shim_and_pybind_build_and_fail_loudly_without_gpu(tmp_path):
    """the drop-in layers compile against the C ABI; without a device they raise, they do not fall back"""
    import subprocess

    lib = os.path.dirname(_capi.LIB_PATH)
    assert os.path.exists(os.path.join(lib, "libopenkitchen_shim.so"))
    csv = tmp_path / "Monza.csv"
    ok.write_track_csv("Monza", str(csv))
    # the checks run in child processes that see no device, so that they also hold on a machine with a GPU
    no_gpu = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([os.path.join(lib, "ok_shim_example"), str(csv), "3", "2"], capture_output=True, text=True, env=no_gpu)
    assert r.returncode != 0 and "no CPU fallback" in r.stderr
    code = ("import open_kitchen_pybind as okp, sys\n"
            "try:\n    okp.Environment(sys.argv[1])\nexcept RuntimeError as ex:\n    print(ex)\n    sys.exit(3)\n")
    r = subprocess.run([sys.executable, "-c", code, str(csv)], cwd=ROOT, capture_output=True, text=True, env=no_gpu)
    assert r.returncode == 3 and "no CPU fallback" in r.stdout, r.stdout + r.stderr


def test_q16_observation_helpers_round_trip():
    """ok_step_host_q16's fixed point, host side: quantise is rn(clamp(obs) * 65535) in binary32 (ties to even), dequantise
    brings every code back to within half a step, and the codes are a fixed point of the round trip."""
    obs = np.array([0.0, 1.0, 0.5, 1.5, -0.25, 0.5 / 65535.0, 1.5 / 65535.0, 2.5 / 65535.0, 0.123456], dtype=np.float32)
    q = ok.quantize_obs_q16(obs)
    assert q.dtype == np.uint16 and list(q[:5]) == [0, 65535, 32768, 65535, 0]
    assert list(q[5:8]) == [0, 2, 2]  # ties to even
    codes = np.arange(65536, dtype=np.uint16)
    back = ok.dequantize_obs_q16(codes)
    assert back.dtype == np.float32 and back[0] == 0.0 and back[-1] == 1.0
    assert np.array_equal(ok.quantize_obs_q16(back), codes)
    rng = np.random.default_rng(0)
    x = rng.random(100000, dtype=np.float32)
    assert np.abs(ok.dequantize_obs_q16(ok.quantize_obs_q16(x)).astype(np.float64) - x).max() <= 0.5 / 65535.0 + 2.0**-22

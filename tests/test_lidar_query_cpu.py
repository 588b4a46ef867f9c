"""CPU: the lidar query's public surface -- the ctypes OkLidarQuery has the C layout, both entry points refuse an env
without a device, and the Python wrappers reject malformed arguments before they reach the library."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

import openkitchen_b200 as ok
from openkitchen_b200 import _capi
from openkitchen_b200.batch_env import BatchEnv

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = [f for f, _ in _capi.OkLidarQuery._fields_]


@pytest.mark.skipif(shutil.which("g++") is None, reason="needs g++")
def test_ctypes_layout_matches_the_header(tmp_path):
    src = tmp_path / "layout.c"
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "openkitchen_b200.h"', "int main(void) {",
             '  printf("%zu\\n", sizeof(OkLidarQuery));']
    lines += [f'  printf("%zu\\n", offsetof(OkLidarQuery, {f}));' for f in FIELDS]
    lines += ["  return 0;", "}"]
    src.write_text("\n".join(lines) + "\n")
    exe = tmp_path / "layout"
    subprocess.run(["g++", "-x", "c++", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert got[0] == C.sizeof(_capi.OkLidarQuery)
    assert got[1:] == [getattr(_capi.OkLidarQuery, f).offset for f in FIELDS]


def test_no_device_means_no_lidar_query():
    with ok.Env(device=-1) as e:
        e.add_named_track("Monza")
        x = np.array([100.0, 200.0], dtype=np.float32)
        with pytest.raises(ok.OkError) as ex:
            e.lidar_query(x, x, x, ray_deg=ok.ray_fan(5))
        assert ex.value.code == _capi.OK_ERR_NO_DEVICE
        with pytest.raises(ok.OkError) as ex:
            e.lidar_query_device(x.ctypes.data, x.ctypes.data, x.ctypes.data, 2, d_ray_deg=x.ctypes.data, rays=2)
        assert ex.value.code == _capi.OK_ERR_NO_DEVICE


def test_env_lidar_query_rejects_bad_arguments_before_the_library():
    with ok.Env(device=-1) as e:  # the library would answer OK_ERR_NO_DEVICE: a ValueError comes from the wrapper
        e.add_named_track("Monza")
        a3, a4 = np.zeros(3, dtype=np.float32), np.zeros(4, dtype=np.float32)
        for args in ((a3, a4, a3), (a3, a3, a4), (a4, a3, a3), (np.zeros((2, 2), dtype=np.float32),) * 3):
            with pytest.raises(ValueError):
                e.lidar_query(*args, ray_deg=ok.ray_fan(5))
        with pytest.raises(ValueError):
            e.lidar_query(a3, a3, a3, track_id=np.zeros(4, dtype=np.int32), ray_deg=ok.ray_fan(5))
        with pytest.raises(ValueError):
            e.lidar_query_device(0, 0, 0, 3, rays=5, observations=0)


class _NoLibrary:
    def __getattr__(self, name):
        raise AssertionError(f"the library was called ({name}) although the arguments are malformed")


def test_batch_env_lidar_rejects_bad_arguments_before_the_library():
    env = BatchEnv.__new__(BatchEnv)  # no device here: only what lidar() reads before its first call
    env.env, env.device, env.n_rays = _NoLibrary(), torch.device("cpu"), 5
    a3, a4 = torch.zeros(3), torch.zeros(4)
    for args in ((a3, a4, a3), (a3, a3, a4), (a4, a3, a3), (torch.zeros(2, 2),) * 3):
        with pytest.raises(ValueError):
            env.lidar(*args)
    with pytest.raises(ValueError):
        env.lidar(a3, a3, a3, track_id=torch.zeros(4, dtype=torch.int32))
    with pytest.raises(ValueError):
        env.lidar(a3, a3, a3, outputs=["obs", "observations"])

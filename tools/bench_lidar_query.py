"""ok_lidar_query against ok_cast_rays on the same poses: prints one JSON line.

Two shapes:
  * bench: bench.py's population (65,536 agents x 32 rays over the 23 tracks, its reset points) after 100 random ticks;
  * latency: 4,096 poses x the 5-ray Q-learning fan on Monza after 100 random ticks.
Per shape, in one process, alternating launch by launch: (a) ok_cast_rays on the population (every crash flag cleared
before the launch, so that every ray is cast), (b) ok_lidar_query on the same poses, reading the population's pos_x /
pos_y / rot / track_id views, all seven outputs.  The L2 is flushed (256 MiB memset) before every timed launch, as in
bench.py; each launch sits between two CUDA events.  The last launch of each arm must agree bit for bit on every output.
The inline share is the beam kernel's debug counter on one extra launch of (a): both arms take the same per-ray decision.

usage: python tools/bench_lidar_query.py [--iters 1000] [--warmup 300]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, limit = (s.strip() for s in out.split(","))
        return name, limit
    except Exception as ex:  # the name from torch, the limit unknown
        import torch

        return torch.cuda.get_device_name(0), f"unavailable ({ex})"


def run_shape(ok, torch, env, n, rays, iters, warmup, flush):
    from openkitchen_b200.dlpack import DeviceBuffer

    v = {nm: torch.from_dlpack(DeviceBuffer(env, nm)) for nm in ok.BUFFERS}
    stream = torch.cuda.current_stream().cuda_stream
    fields = {"obs": (n, rays), "hit_rel": (n, rays, 2), "hit_abs": (n, rays, 2), "hit_t": (n, rays), "hit_seg": (n, rays),
              "min_dist2": (n,), "crashed": (n,)}
    dtypes = {"hit_seg": torch.int32, "crashed": torch.uint8}
    out = {f: torch.empty(s, device="cuda", dtype=dtypes.get(f, torch.float32)) for f, s in fields.items()}
    ptrs = {f: t.data_ptr() for f, t in out.items()}

    def cast():
        v["crashed"].zero_()
        env.cast_rays(stream)

    def query():
        env.lidar_query_device(v["pos_x"].data_ptr(), v["pos_y"].data_ptr(), v["rot"].data_ptr(), n, v["track_id"].data_ptr(),
                               None, rays, stream, **ptrs)

    for _ in range(warmup):  # past the feedback tiling's re-cuts (launches 16, 64 and 256 of ok_cast_rays)
        cast()
        query()
    torch.cuda.synchronize()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(iters)]
    for e in ev:
        flush.zero_()
        v["crashed"].zero_()
        e[0].record()
        env.cast_rays(stream)
        e[1].record()
        flush.zero_()
        e[2].record()
        query()
        e[3].record()
    torch.cuda.synchronize()
    ta = np.array([e[0].elapsed_time(e[1]) for e in ev])
    tb = np.array([e[2].elapsed_time(e[3]) for e in ev])
    same = {f: bool(((v[f].view(torch.int32) == out[f].view(torch.int32)) | (torch.isnan(v[f]) & torch.isnan(out[f]))).all())
            if out[f].dtype == torch.float32 else bool(torch.equal(v[f], out[f])) for f in fields}
    assert all(same.values()), f"the two arms differ: {same}"
    env.debug_stats(True)
    cast()
    cast_n, queued, walked = env.debug_stats(False)
    res = {"poses": n, "rays": rays, "launches_per_arm": iters,
           "cast_rays_ms": round(float(ta.mean()), 5), "cast_rays_ms_median": round(float(np.median(ta)), 5),
           "lidar_query_ms": round(float(tb.mean()), 5), "lidar_query_ms_median": round(float(np.median(tb)), 5),
           "cast_rays_rays_per_s": n * rays / (ta.mean() * 1e-3), "lidar_query_rays_per_s": n * rays / (tb.mean() * 1e-3),
           "bit_identical": True}
    if cast_n:
        res["inline_share"] = round(1.0 - queued / cast_n, 5)
        res["grid_walk_share"] = round(walked / cast_n, 6)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=300)
    args = ap.parse_args()
    import torch

    import openkitchen_b200 as ok
    from bench import N_AGENTS, N_RAYS, build_workload

    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    env = ok.Env(device=0, movement_mode=ok.MOVE_VELOCITY, reward_mode=ok.REWARD_CMAES_PROGRESS, auto_reset=1)
    build_workload(ok, env, N_AGENTS)
    env.launch_steps_random(0, 100)
    bench = run_shape(ok, torch, env, N_AGENTS, N_RAYS, args.iters, args.warmup, flush)
    env.close()
    env = ok.Env(device=0, movement_mode=ok.MOVE_VELOCITY, reward_mode=ok.REWARD_Q_PROGRESS, auto_reset=1)
    env.add_named_track("Monza")
    env.alloc_agents(4096, np.array([-70, -30, 0, 30, 70], dtype=np.float32))
    env.reset(None, (np.arange(4096) * 2654435761 % 2**32 % env.track_info(0).n_points).astype(np.int32))
    env.launch_steps_random(0, 100)
    latency = run_shape(ok, torch, env, 4096, 5, args.iters, args.warmup, flush)
    env.close()
    name, limit = card()
    print(json.dumps({"tool": "bench_lidar_query", "gpu": name, "power_limit": limit,
                      "l2": "flushed before every timed launch (256 MiB memset)", "timing": "CUDA events around each launch",
                      "bench_shape": bench, "latency_shape": latency}))


if __name__ == "__main__":
    main()

"""ok_bev_query (bird's-eye-view rasters) against one ok_cast_rays of the same population: prints one JSON line.

Three shapes:
  * silverstone: 4,096 poses x 64x64, scale 1, on Silverstone after 100 random ticks;
  * bench: bench.py's population (65,536 agents x 32 rays over the 23 tracks, its reset points) after 100 random ticks,
    x 64x64, scale 1;
  * wide: the Silverstone population x 96x96, scale 2, ahead 32.
Per shape, in one process, alternating launch by launch: (a) ok_cast_rays on the population (every crash flag cleared
before the launch, so that every ray is cast), (b) ok_bev_query at the population's poses, reading its pos_x / pos_y /
rot / track_id views.  The L2 is flushed (256 MiB memset) before every timed launch, as in bench.py; each launch sits
between two CUDA events.  Reported per shape: ms per call, pixels per second, output bytes over time against the
7.7 TB/s HBM write floor of the data sheet, and the time of (b) over (a).

usage: python tools/bench_bev.py [--iters 300] [--warmup 50]
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.bench_lidar_query import card  # noqa: E402

HBM_BYTES_PER_S = 7.7e12  # B200 data sheet (one GPU of an HGX B200)


def run_shape(ok, torch, env, n, h, w, scale, ahead, iters, warmup, flush):
    from openkitchen_b200.dlpack import DeviceBuffer

    v = {nm: torch.from_dlpack(DeviceBuffer(env, nm)) for nm in ("pos_x", "pos_y", "rot", "track_id", "crashed")}
    stream = torch.cuda.current_stream().cuda_stream
    out = torch.empty((n, h, w), dtype=torch.uint8, device="cuda")

    def cast():
        v["crashed"].zero_()
        env.cast_rays(stream)

    def query():
        env.bev_query_device(v["pos_x"].data_ptr(), v["pos_y"].data_ptr(), v["rot"].data_ptr(), n, h, w, scale,
                             out.data_ptr(), ahead, v["track_id"].data_ptr(), stream)

    for _ in range(warmup):
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
    px = n * h * w
    frac = np.bincount(out.view(-1).cpu().numpy(), minlength=3) / px
    return {"poses": n, "height": h, "width": w, "scale": scale, "ahead": ahead, "launches_per_arm": iters,
            "bev_ms": round(float(tb.mean()), 5), "bev_ms_median": round(float(np.median(tb)), 5),
            "cast_rays_ms": round(float(ta.mean()), 5), "cast_rays_ms_median": round(float(np.median(ta)), 5),
            "pixels_per_s": px / (tb.mean() * 1e-3), "output_bytes": px,
            "write_floor_share": round(px / HBM_BYTES_PER_S / (tb.mean() * 1e-3), 5),
            "bev_over_cast_rays": round(float(tb.mean() / ta.mean()), 4),
            "class_shares": {"off": round(float(frac[0]), 4), "wall": round(float(frac[1]), 4), "lane": round(float(frac[2]), 4)}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=50)
    args = ap.parse_args()
    import torch

    import openkitchen_b200 as ok
    from bench import N_AGENTS, N_RAYS, build_workload

    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    env = ok.Env(device=0, movement_mode=ok.MOVE_VELOCITY, reward_mode=ok.REWARD_CMAES_PROGRESS, auto_reset=1)
    env.add_named_track("Silverstone")
    env.alloc_agents(4096, ok.ray_fan(N_RAYS))
    env.reset(None, (np.arange(4096) * 2654435761 % 2**32 % env.track_info(0).n_points).astype(np.int32))
    env.launch_steps_random(0, 100)
    silverstone = run_shape(ok, torch, env, 4096, 64, 64, 1.0, 0.0, args.iters, args.warmup, flush)
    wide = run_shape(ok, torch, env, 4096, 96, 96, 2.0, 32.0, args.iters, args.warmup, flush)
    env.close()
    env = ok.Env(device=0, movement_mode=ok.MOVE_VELOCITY, reward_mode=ok.REWARD_CMAES_PROGRESS, auto_reset=1)
    build_workload(ok, env, N_AGENTS)
    env.launch_steps_random(0, 100)
    bench = run_shape(ok, torch, env, N_AGENTS, 64, 64, 1.0, 0.0, args.iters, args.warmup, flush)
    env.close()
    name, limit = card()
    print(json.dumps({"tool": "bench_bev", "gpu": name, "power_limit": limit,
                      "l2": "flushed before every timed launch (256 MiB memset)", "timing": "CUDA events around each launch",
                      "write_floor": "output bytes / 7.7e12 B/s over the measured time", "silverstone_shape": silverstone,
                      "bench_shape": bench, "wide_shape": wide}))


if __name__ == "__main__":
    main()

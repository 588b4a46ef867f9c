"""Lap accounting on against off at bench.py's shape: prints one JSON line.

Two envs built like bench.py's (65,536 agents x 32 rays over the 23 tracks, VELOCITY mode, random Philox actions,
auto-reset), one with lap accounting off and one with it on at target 0 (laps are counted, no agent completes), so both
arms drive the same agents through the same states and differ only in the accounting.  After --warmup ticks each, the two
are timed alternately, one tick at a time, each tick between two CUDA events with the L2 flushed (256 MiB memset) before
it, as in bench.py.  --reward picks the reward mode: the accounting needs the nearest centre-line index every tick, which
the progress modes (1, 2, 6, 7; bench.py's is 2) search anyway and the others (3-5) do not.

usage: python tools/bench_laps.py [--iters 600] [--warmup 300] [--reward 2]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=600)
    ap.add_argument("--warmup", type=int, default=300)
    ap.add_argument("--reward", type=int, default=2)
    args = ap.parse_args()
    import torch

    import openkitchen_b200 as ok
    from bench import N_AGENTS, SEED, build_workload

    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    envs = {}
    for arm in ("off", "on"):
        env = ok.Env(device=0, movement_mode=ok.MOVE_VELOCITY, reward_mode=args.reward, auto_reset=1)
        build_workload(ok, env, N_AGENTS)
        if arm == "on":
            env.set_laps(0)
        env.launch_steps_random(0, args.warmup, SEED)
        envs[arm] = env
    torch.cuda.synchronize()
    ms = {arm: [] for arm in envs}
    crashed = {arm: [] for arm in envs}
    stream = torch.cuda.current_stream().cuda_stream
    for i in range(args.iters):
        for arm, env in envs.items():
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            env.launch_steps_random(args.warmup + i, 1, SEED, stream)
            b.record()
            b.synchronize()
            ms[arm].append(a.elapsed_time(b))
            if i % 50 == 0:
                crashed[arm].append(env.population_counters(stream)["crashed"])
    info = envs["on"].lap_buffers_info()["laps"]
    laps = torch.from_dlpack(ok.dlpack.DeviceBuffer(envs["on"], "laps", info)).to(torch.int64)
    name, limit = card()
    out = {"tool": "bench_laps", "reward_mode": args.reward, "gpu": name, "power_limit": limit, "agents": N_AGENTS, "iters": args.iters,
           "l2": "flushed before every timed tick (256 MiB memset)", "timing": "CUDA events around each tick, arms alternating"}
    for arm in envs:
        v = sorted(ms[arm])
        out[arm] = {"median_ms": statistics.median(v), "p10_ms": v[len(v) // 10], "p90_ms": v[9 * len(v) // 10],
                    "mean_crashed_per_tick": statistics.mean(crashed[arm])}
    out["laps_counted"] = int(laps.sum())
    out["on_over_off_median"] = out["on"]["median_ms"] / out["off"]["median_ms"]
    print(json.dumps(out))


if __name__ == "__main__":
    main()

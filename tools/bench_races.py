"""Races off against on: prints one JSON line.

Part 1, bench.py's shape: one env built like bench.py's (65,536 agents x 32 rays over the 23 tracks, VELOCITY mode, random
Philox actions, auto-reset).  After --warmup ticks, the arms -- races off, then on with group 2, 8, 32, 256 and 1,024 --
take one tick each in turn, in the same process and on the same env (ok_set_races between ticks), each tick between two
CUDA events with the L2 flushed (256 MiB memset) before it, as in bench.py.  The agents start spread over their tracks, as
in bench.py, so most opponents are out of lidar range: the cull decides most pairs.

Part 2, config 4 (PPO rollout collection, tools/bench_c4.py: 4,096 agents on Monza, 5 rays, actor 5-128-3): two
FusedActorRollouts of --steps ticks captured as CUDA graphs, one env with races off and one with group 8, replayed
alternately with the L2 flushed before each replay; ms per tick = replay time / steps.

usage: python tools/bench_races.py [--iters 300] [--warmup 200] [--radius 4] [--steps 64] [--replays 20]
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

GROUPS = (2, 8, 32, 256, 1024)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, limit = (s.strip() for s in out.split(","))
        return name, limit
    except Exception as ex:  # the name from torch, the limit unknown
        import torch

        return torch.cuda.get_device_name(0), f"unavailable ({ex})"


def stats(v):
    v = sorted(v)
    return {"median_ms": statistics.median(v), "p10_ms": v[len(v) // 10], "p90_ms": v[9 * len(v) // 10]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--radius", type=float, default=4.0)
    ap.add_argument("--steps", type=int, default=64)
    ap.add_argument("--replays", type=int, default=20)
    args = ap.parse_args()
    import torch

    import openkitchen_b200 as ok
    from bench import N_AGENTS, SEED, build_workload
    from openkitchen_b200.rollout import FusedActorRollout

    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")
    stream = torch.cuda.current_stream().cuda_stream

    def timed(fn):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        return a.elapsed_time(b)

    # ---- part 1: bench.py's shape ----
    env = ok.Env(device=0, movement_mode=ok.MOVE_VELOCITY, reward_mode=ok.REWARD_CMAES_PROGRESS, auto_reset=1)
    build_workload(ok, env, N_AGENTS)
    arms = (0,) + GROUPS
    tick = 0
    for g in arms:  # every arm warmed up (the first launch of the pass loads its module)
        env.set_races(g, args.radius)
        env.launch_steps_random(tick, args.warmup // len(arms) + 1, SEED, stream)
        tick += args.warmup // len(arms) + 1
    torch.cuda.synchronize()
    ms = {g: [] for g in arms}
    contacts = {g: 0 for g in GROUPS}
    for i in range(args.iters):
        for g in arms:
            env.set_races(g, args.radius)
            ms[g].append(timed(lambda: env.launch_steps_random(tick, 1, SEED, stream)))
            tick += 1
            if g and i % 50 == 0:
                contacts[g] += int(torch.from_dlpack(ok.dlpack.DeviceBuffer(env, "contact", env.race_buffers_info()["contact"])).sum())
    name, limit = card()
    out = {"tool": "bench_races", "gpu": name, "power_limit": limit, "agents": N_AGENTS, "rays": env.rays, "tracks": env.num_tracks(),
           "radius": args.radius, "iters": args.iters, "l2": "flushed before every timed tick or replay (256 MiB memset)",
           "timing": "CUDA events around each tick, arms alternating on one env"}
    out["off"] = stats(ms[0])
    for g in GROUPS:
        out[f"group_{g}"] = dict(stats(ms[g]), added_median_ms=statistics.median(ms[g]) - out["off"]["median_ms"],
                                 contact_crashes_sampled=contacts[g])
    env.close()

    # ---- part 2: config 4's FusedActorRollout tick, races off and group 8 ----
    torch.manual_seed(0)
    l1, l2 = torch.nn.Linear(5, 128).cuda(), torch.nn.Linear(128, 3).cuda()
    table = torch.tensor([[60.0, 0.0], [60.0, -3.0], [60.0, 3.0]], device="cuda")
    rolls = {}
    for g in (0, 8):
        be = ok.BatchEnv(["Monza"], 4096, rays=[-70, -30, 0, 30, 70], reward_mode=ok.REWARD_CONSTANT, auto_reset=1)
        be.set_races(g, args.radius)
        fr = FusedActorRollout(be, l1, l2, table, args.steps, sample=True)
        be.reset_random()
        be.cast_rays()
        fr.capture()
        fr.run()
        rolls[g] = (be, fr)
    torch.cuda.synchronize()
    c4 = {g: [] for g in rolls}
    for _ in range(args.replays):
        for g, (_, fr) in rolls.items():
            c4[g].append(timed(fr.run) / args.steps)
    out["config4_fused_actor"] = {"agents": 4096, "rays": 5, "steps_per_replay": args.steps, "off": stats(c4[0]),
                                  "group_8": stats(c4[8]),
                                  "group_8_done_fraction": float(rolls[8][1].dones.float().mean()),
                                  "off_done_fraction": float(rolls[0][1].dones.float().mean())}
    print(json.dumps(out))


if __name__ == "__main__":
    main()

#!/usr/bin/env python
"""bench.py -- agent-steps/s and ray-casts/s of the batched step loop on B200 (BASELINE.json metric).

    python bench.py --gpus 1 --steps 1000 --warmup 100            # our arm (N>1: under torchrun)
    python bench.py --impl reference --steps K --warmup W          # the reference CPU arm

Workload (BASELINE.json configs[2], the shape the 1e10 ray-casts/s target is quoted on): 65,536
agents spread over all 23 tracks, 32 rays each, random (Philox) actions, VELOCITY mode, crashed
agents auto-reset, CMA-ES progress reward (nearest centre-line index every tick).  A "step" is one
tick of every agent.  At N GPUs every rank owns its own 65,536-agent slice (weak scaling, no
data-path collective: agents never interact).

Timing: W warm-up ticks, then K ticks each bracketed by CUDA events on the launching stream with an
L2 flush (a 256 MiB memset) between ticks; ms_per_step = mean event time, max over ranks.  The
`e2e` number drives the same tick through ok_step_host with pinned HOST buffers (H2D actions, D2H
obs/reward/done inside the timed region).

`--dump-outputs DIR` writes the buffers the last timed tick left (observations, rewards, flags, poses, ...) as
DIR/<name>.npy, so that two builds can be compared output for output on identical inputs.  At N GPUs it writes rank 0's
slice of the population only.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_AGENTS = 65536
N_RAYS = 32
SEED = 0x0C17C4E2
BYTES_PER_AGENT_STEP = 92 + 8 * N_RAYS  # SURVEY.md 8(d): 348 B at R = 32
WORKLOAD = "C3: 65536 agents over 23 tracks x 32 rays, random actions, auto-reset, progress reward"


def ncu_evidence():
    """DRAM traffic per launch of the step kernel from the committed `ncu --set full` capture (profiles/)."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        return json.load(open(p))
    except Exception:
        return None


def peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "25", "-i", str(self.index)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax = float(f[2])
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


SETTLE_TICKS = 80  # launches before the timed region (warm-up included): the library's feedback tiling has settled by then


def build_workload(ok, env_or_oracle, n_agents, is_oracle=False, id_base=0, period=None, n_total=None):
    """tracks + agents + deterministic reset of SURVEY 8(d); identical for the product and the oracle.
    `id_base`: this env holds the agents [id_base, id_base + n_agents) of a larger population (a rank's shard, or a
    slice replayed alone).  The reset point is a function of the GLOBAL agent id; the track is a function of the id
    modulo `period` (default n_agents; n_total is an alias): every `period` consecutive agents -- one GPU's slice in the
    weak-scaling runs -- are spread over all 23 tracks."""
    names = ok.track_names()
    pts_per_track = []
    for nm in names:
        cols = ok.track_columns(nm)
        if is_oracle:
            env_or_oracle.add_track(cols)
        else:
            env_or_oracle.add_track(cols)
        pts_per_track.append(len(cols[0]))
    nt = len(names)
    period = period if period is not None else (n_total if n_total is not None else n_agents)
    gid = np.arange(id_base, id_base + n_agents, dtype=np.int64)
    tid = ((gid % period) * nt // period).astype(np.int32)  # contiguous per track
    env_or_oracle.alloc_agents(n_agents, ok.ray_fan(N_RAYS), tid)
    ids = gid.astype(np.uint64)
    pts = ((ids * np.uint64(2654435761)) % np.uint64(2**32) % np.asarray(pts_per_track, dtype=np.uint64)[tid]).astype(np.int32)
    env_or_oracle.reset(None, pts)
    return tid


def cpu_reference_run(steps, warmup, budget_s, n_cap=N_AGENTS):
    """Times the reference CPU implementation (oracle/_ref when built, else the C port) with every
    host thread on a bounded sample of the workload.  Returns (agent_steps_per_s, info dict)."""
    import openkitchen_b200 as ok
    from oracle import api as oapi

    kind = "reference" if oapi.have_ref() else "port"
    cfg = dict(movement_mode=0, reward_mode=2, auto_reset=1)
    # calibration tick on a small sample to size the run
    cal = oapi.Oracle(kind, **cfg)
    cores = cal.max_threads()
    cal.set_threads(cores)
    n_cal = 23 * 8
    build_workload(ok, cal, n_cal, is_oracle=True)
    cal.fill_random_actions(0, SEED)
    cal.step()
    t0 = time.perf_counter()
    for s in range(1, 4):
        cal.fill_random_actions(s, SEED)
        cal.step()
    rate = 3 * n_cal / (time.perf_counter() - t0)
    cal.close()
    total_ticks = max(1, steps + warmup)
    n = int(min(n_cap, max(23, rate * budget_s / total_ticks)))
    n = max(23, (n // 23) * 23)
    ora = oapi.Oracle(kind, **cfg)
    ora.set_threads(cores)
    build_workload(ok, ora, n, is_oracle=True)
    for s in range(warmup):
        ora.fill_random_actions(s, SEED)
        ora.step()
    t0 = time.perf_counter()
    for s in range(warmup, warmup + steps):
        ora.fill_random_actions(s, SEED)
        ora.step()
    dt = time.perf_counter() - t0
    ora.close()
    value = n * steps / dt
    info = {"value": value, "unit": "agent-steps/s", "cores": cores, "kind": kind,
            "sample": f"{n} agents (same 23-track mix, ray fan, Philox actions, auto-reset) x {steps} ticks after {warmup} warm-up, {dt:.1f} s"}
    return value, dt, info


def ref_cuda_kernel_baseline(ok, n=4096, iters=30):
    """Secondary baseline: the reference's REAL CollisionChecker (its CUDA kernel + per-step Ray_ H2D/D2H memcpys +
    host pack/unpack loops, CollisionChecker.cu:113-174) compiled unchanged for sm_100a, on this GPU, at BASELINE
    config 1's shape (4,096 agents x 32 rays on Silverstone; the reference's uint16_t loop caps it below 65,536)."""
    import ctypes as C
    import tempfile

    lib = os.path.join(ROOT, "oracle", "_ref", "libokref_cuda.so")
    if not os.path.exists(lib):
        return None
    ref = C.CDLL(lib)
    ref.okc_create.restype = C.c_void_p
    ref.okc_create.argtypes = [C.c_char_p, C.c_int64, C.c_int, C.c_void_p]
    ref.okc_set_poses.argtypes = [C.c_void_p] * 5
    ref.okc_time_checks.restype = C.c_double
    ref.okc_time_checks.argtypes = [C.c_void_p, C.c_int]
    ref.okc_destroy.argtypes = [C.c_void_p]
    fan = ok.ray_fan(N_RAYS)
    with tempfile.TemporaryDirectory() as d:
        csv = os.path.join(d, "Silverstone.csv")
        ok.write_track_csv("Silverstone", csv)
        env = ok.Env(device=-1)
        t = env.add_named_track("Silverstone")
        tx, ty, th = env.track_array(t, "x"), env.track_array(t, "y"), env.track_array(t, "heading")
        idx = (np.arange(n, dtype=np.int64) * 2654435761 % 2**32 % len(tx)).astype(np.int64)
        x, y, rot = tx[idx].copy(), ty[idx].copy(), th[idx].copy()
        h = ref.okc_create(csv.encode(), n, N_RAYS, fan.ctypes.data_as(C.c_void_p))
        ref.okc_set_poses(h, x.ctypes.data_as(C.c_void_p), y.ctypes.data_as(C.c_void_p), rot.ctypes.data_as(C.c_void_p), None)
        ref.okc_time_checks(h, 3)
        sec = ref.okc_time_checks(h, iters)
        ref.okc_destroy(h)
    return {"what": "reference CollisionChecker::checkCollision (raycast + memcpys + host loops only, no kinematics), sm_100a build",
            "agents": n, "rays": N_RAYS, "track": "Silverstone", "ms_per_check": 1e3 * sec / iters,
            "ray_casts_per_sec": n * N_RAYS * iters / sec}


def workload_config(n, world):
    """the `config` object: identical for our arm and the reference arm (it names the workload, not the implementation)"""
    return {"workload": WORKLOAD, "agents_per_gpu": n, "rays": N_RAYS, "tracks": 23, "movement": "VELOCITY",
            "actions": "Philox4x32-10 keyed by (global agent id, tick)", "reward": "CMA-ES progress (nearest centre-line index every tick)",
            "auto_reset": True, "parallelism": f"agent-sharded x{world}, no per-tick collective",
            "l2": "GPU arm: flushed between timed ticks (256 MiB memset)"}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    value, dt, info = cpu_reference_run(args.steps, args.warmup, budget_s=90.0)
    line = {
        "impl": "reference", "metric": "agent_steps_per_sec", "value": value, "unit": "agent-steps/s",
        "ray_casts_per_sec": value * N_RAYS, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dt / max(1, args.steps), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": workload_config(args.agents, max(world, args.gpus)),
        "impl_config": {"note": "CPU arm: each step is one tick of a bounded agent sample of the workload, all host threads"},
        "cpu_baseline": info,
        "e2e": {"value": value, "unit": "agent-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


class NvmlSampler:
    """SM clock / throttle reasons sampled IN PROCESS through NVML every few ms (the nvidia-smi loop of round 1 gave
    0-1 samples over a 30 ms timed region).  Falls back to the nvidia-smi loop when pynvml is missing."""

    HW_SLOWDOWN, SW_POWER_CAP, SW_THERMAL, HW_THERMAL = 0x8, 0x4, 0x20, 0x40

    def __init__(self, torch, local: int, period_s: float = 0.004):
        self.period, self.samples, self.power, self.reasons = period_s, [], [], 0
        self.stop_flag = threading.Event()
        self.fallback = None
        self.marks = {}
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            props = torch.cuda.get_device_properties(local)
            try:
                bus = "%08x:%02x:%02x.0" % (props.pci_domain_id, props.pci_bus_id, props.pci_device_id)
                self.h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
            except Exception:
                vis = os.environ.get("CUDA_VISIBLE_DEVICES")
                idx = int(vis.split(",")[local]) if vis and vis.split(",")[local].isdigit() else local
                self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.smax = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None
            self.fallback = ClockSampler(local)

    def start(self):
        if self.nv is None:
            self.fallback.start()
            return
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()

    def _run(self):
        nv = self.nv
        while not self.stop_flag.is_set():
            try:
                self.samples.append((time.perf_counter(), float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))))
                self.reasons |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
            except Exception:
                pass
            time.sleep(self.period)

    def mark(self, name):
        self.marks[name] = time.perf_counter()

    def stop(self):
        if self.nv is None:
            return self.fallback.stop()
        self.stop_flag.set()
        self.t.join(timeout=1.0)
        t0, t1 = self.marks.get("timed_begin", 0.0), self.marks.get("timed_end", float("inf"))
        timed = [c for t, c in self.samples if t0 <= t <= t1]
        allc = [c for _, c in self.samples]
        reasons = [n for n, bit in (("hw_slowdown", self.HW_SLOWDOWN), ("hw_thermal_slowdown", self.HW_THERMAL),
                                    ("sw_thermal_slowdown", self.SW_THERMAL), ("sw_power_cap", self.SW_POWER_CAP)) if self.reasons & bit]
        return {"sm_mhz": float(np.median(timed if timed else allc)) if allc else None, "sm_max_mhz": self.smax, "reasons": reasons,
                "samples": len(allc), "samples_in_timed_region": len(timed), "sm_mhz_min": min(allc) if allc else None,
                "window_s": (self.samples[-1][0] - self.samples[0][0]) if len(self.samples) > 1 else 0.0,
                "power_w_max": max(self.power) if self.power else None, "source": "NVML in-process, %.0f ms period" % (1e3 * self.period)}


def bind_to_gpu_numa_node(torch, local: int):
    """Pin this rank's host threads (and therefore the pinned buffers it allocates from now on: first touch) to the NUMA
    node its GPU hangs off, so that the end-to-end path's PCIe traffic does not cross the socket interconnect."""
    try:
        props = torch.cuda.get_device_properties(local)
        bus = "%04x:%02x:%02x.0" % (props.pci_domain_id, props.pci_bus_id, props.pci_device_id)
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read().strip())
        if node < 0:
            return {"numa_node": None, "note": "no NUMA information for the GPU"}
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.extend(range(int(a), int(b or a) + 1))
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if not allowed:
            return {"numa_node": node, "note": "node's CPUs are outside this process's affinity mask"}
        os.sched_setaffinity(0, allowed)
        return {"numa_node": node, "cpus": len(allowed)}
    except Exception as ex:
        return {"numa_node": None, "note": f"not bound: {ex}"}


PARITY_BUFS = ("pos_x", "pos_y", "rot", "crashed", "timed_out", "hit_seg", "hit_t", "obs", "reward", "fitness", "nearest_idx", "reset_pt")
DUMP_BUFS = PARITY_BUFS + ("speed", "done")
DUMP_BYTES = 60_000_000  # array data; with the .npy headers the files stay under 64 MB


def dump_outputs(env, directory, stream=None):
    """--dump-outputs: the buffers a caller of the tick reads, as DIR/<name>.npy.  binary32 buffers as they are, flags as
    float32 and indices as float64 (both exact).  A population whose buffers would exceed DUMP_BYTES is cut to a fixed,
    seeded sample of agents, the same rows in every buffer; agent_index.npy then names those rows."""
    arrays = {}
    for name in DUMP_BUFS:
        a = env.read(name, stream)
        arrays[name] = a.astype(np.float64 if a.dtype.kind in "iu" and a.itemsize == 4 else np.float32)
    rows = None
    per_agent = sum(a.nbytes for a in arrays.values()) // env.n
    if per_agent * env.n > DUMP_BYTES:
        k = DUMP_BYTES // (per_agent + 8)
        rows = np.sort(np.random.default_rng(SEED).choice(env.n, k, replace=False))
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, f"{name}.npy"), a if rows is None else a[rows])
    if rows is not None:
        np.save(os.path.join(directory, "agent_index.npy"), rows.astype(np.float64))


def shard_parity_check(ok, torch, dist, env, rank, n, ticks, local, mode, extra):
    """N > 1: rank 0 replays, alone and from scratch, the first 1,024 agents of rank 1's slice (global ids n .. n+1023)
    and compares every listed buffer bit for bit with what rank 1 computed inside its 65,536-agent shard."""
    m = min(1024, n)
    packed = None
    if rank == 1:
        parts = [np.ascontiguousarray(env.read(b)[:m]).view(np.uint8).reshape(-1) for b in PARITY_BUFS]
        packed = torch.from_numpy(np.concatenate(parts)).cuda()
        dist.send(packed, dst=0)
        return None
    if rank != 0:
        return None
    twin = ok.Env(device=local, movement_mode=ok.MOVE_VELOCITY, reward_mode=ok.REWARD_CMAES_PROGRESS, auto_reset=1,
                  raycast_mode=mode, agent_id_base=n, **extra)
    build_workload(ok, twin, m, id_base=n, period=n)
    twin.launch_steps_random(0, ticks, SEED)
    twin.sync()
    parts = [np.ascontiguousarray(twin.read(b)).view(np.uint8).reshape(-1) for b in PARITY_BUFS]
    mine = np.concatenate(parts)
    twin.close()
    theirs = torch.empty(mine.size, dtype=torch.uint8, device="cuda")
    dist.recv(theirs, src=1)
    theirs = theirs.cpu().numpy()
    if np.array_equal(mine, theirs):
        return "ok"
    off = 0
    for b, part in zip(PARITY_BUFS, parts):
        if not np.array_equal(part, theirs[off:off + part.size]):
            return f"MISMATCH in {b}"
        off += part.size
    return "MISMATCH"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=100)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--agents", type=int, default=N_AGENTS, help="agents per GPU (default: the BASELINE workload)")
    ap.add_argument("--raycast", default="beam", choices=["beam", "grid", "brute"])
    ap.add_argument("--beam-cell", type=float, default=0.0, help="beam table start-cell size in px (0 = library default)")
    ap.add_argument("--beam-bins", type=int, default=0, help="beam table direction bins (0 = library default)")
    ap.add_argument("--cell", type=float, default=0.0, help="broadphase cell size in px (0 = library default)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-flush", action="store_true", help="do not flush L2 between timed ticks")
    ap.add_argument("--generation", type=int, default=100, help="N>1: ticks between two fitness exchanges (NCCL all-gather + ranking)")
    ap.add_argument("--no-numa", action="store_true", help="do not bind the rank to its GPU's NUMA node")
    ap.add_argument("--config5", action="store_true", help="also run BASELINE configs[4]'s shape: 1,048,576 agents per GPU + CMA-ES exchange")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the buffers of the last timed tick as DIR/<name>.npy (float32 / float64, at most 64 MB; rank 0's agents)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU arm's buffers: it needs --impl ours")
    args.warmup = max(args.warmup, 3)

    if args.impl == "reference":
        run_reference_arm(args)
        return

    import torch

    import openkitchen_b200 as ok

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: openkitchen_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    numa = {"numa_node": None, "note": "disabled"} if args.no_numa else bind_to_gpu_numa_node(torch, local)
    dist = None
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    n = args.agents
    extra = {"grid_cell": args.cell} if args.cell > 0 else {}
    if args.beam_cell > 0:
        extra["beam_cell"] = args.beam_cell
    if args.beam_bins > 0:
        extra["beam_bins"] = args.beam_bins
    mode = {"beam": ok.RAYCAST_BEAM, "grid": ok.RAYCAST_GRID, "brute": ok.RAYCAST_BRUTE}[args.raycast]
    # every rank owns the agents [rank * n, (rank + 1) * n) of the global population: Philox stream and reset points are
    # functions of the GLOBAL id (OkConfig::agent_id_base), so the sharded run is the unsharded run, slice by slice
    env = ok.Env(device=local, movement_mode=ok.MOVE_VELOCITY, reward_mode=ok.REWARD_CMAES_PROGRESS, auto_reset=1,
                 raycast_mode=mode, agent_id_base=rank * n, **extra)
    t_build = time.perf_counter()
    build_workload(ok, env, n, id_base=rank * n, period=n)
    env.cast_rays(None)  # first launch uploads the track arena (and builds the beam tables): outside every timed region
    env.sync()
    t_build = time.perf_counter() - t_build
    table_bytes = sum(env.beam_table_bytes(t) for t in range(env.num_tracks())) if mode == ok.RAYCAST_BEAM and rank == 0 else None
    stream = torch.cuda.current_stream()
    sp = stream.cuda_stream
    flush = None if args.no_flush else torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    # ---- sharded == unsharded (N > 1), on the first ticks after the reset; these ticks double as warm-up ----------
    parity_ticks = 50
    shard_parity = None
    step_base = 0
    if dist is not None:
        env.launch_steps_random(0, parity_ticks, SEED, sp)
        env.sync(sp)
        shard_parity = shard_parity_check(ok, torch, dist, env, rank, n, parity_ticks, local, mode, extra)
        step_base = parity_ticks

    # ---- device-resident arm ----------------------------------------------------------------
    for s in range(args.warmup):
        env.launch_steps_random(step_base + s, 1, SEED, sp)
    step_base += args.warmup
    # The library re-cuts its tiles from measured tile times after the 16th and the 64th launch of an env (feedback tiling,
    # ok_balance_schedule): a warm-up shorter than that is topped up, untimed and under the timed region's conditions (L2
    # flushed between ticks), so that the timed ticks see the schedule of any run longer than a second's worth of ticks.
    settle = max(0, SETTLE_TICKS - (step_base if dist is not None else args.warmup)) if mode == ok.RAYCAST_BEAM else 0
    for s in range(settle):
        if flush is not None:
            flush.zero_()
        env.launch_steps_random(step_base + s, 1, SEED, sp)
    step_base += settle
    fit_view = torch.from_dlpack(ok.dlpack.DeviceBuffer(env, "fitness"))
    gen_every = max(1, args.generation)
    if dist is not None:  # warm the communicator and the sort outside the timed region
        from openkitchen_b200 import dist as okdist

        for _ in range(2):
            okdist.global_ranking(fit_view, n * world)
    barrier()
    launches0 = env.launch_stats().kernel_launches
    sampler = NvmlSampler(torch, local)
    if rank == 0:
        sampler.start()
        sampler.mark("timed_begin")
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    stops = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    gens = []
    t_wall = time.perf_counter()
    for i in range(args.steps):
        if flush is not None:
            flush.zero_()
        starts[i].record(stream)
        env.launch_steps_random(step_base + i, 1, SEED, sp)
        stops[i].record(stream)
        if dist is not None and (i + 1) % gen_every == 0:
            # the generation boundary of the population learners: every rank needs every candidate's fitness and the
            # same ranking (CmaEsSolverTorch.cpp:81-96, Mating.hpp:108-119) -- the ONLY exchange on the data path
            g0, gm, g1 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            g0.record(stream)
            gathered = okdist.all_gather_fitness(fit_view, n * world)  # NCCL over NVLink
            gm.record(stream)
            torch.sort(gathered, descending=True, stable=True)        # the ranking every rank derives (ties by global id)
            g1.record(stream)
            gens.append((g0, g1, gm))
    barrier()
    t_wall = time.perf_counter() - t_wall
    if rank == 0:
        sampler.mark("timed_end")
    launches = env.launch_stats().kernel_launches - launches0
    ms = np.array([a.elapsed_time(b) for a, b in zip(starts, stops)], dtype=np.float64)
    ms_tick = float(ms.mean())
    gen_ms = float(np.mean([a.elapsed_time(b) for a, b, _ in gens])) if gens else 0.0
    gather_ms = float(np.mean([a.elapsed_time(m) for a, _, m in gens])) if gens else 0.0
    ms_per_step = ms_tick + gen_ms * len(gens) / args.steps
    crashed_frac = float(env.read("crashed", sp).mean())
    if args.dump_outputs and rank == 0:
        dump_outputs(env, args.dump_outputs, sp)
    step_base += args.steps
    # clock window: the timed region of a short run is a few ms; keep the same launches going (untimed) until the
    # sampler has seen >= 1 s of this workload
    if rank == 0:
        t_end = time.perf_counter() + max(0.0, 1.0 - t_wall)
        k = 0
        while time.perf_counter() < t_end:
            env.launch_steps_random(step_base + k, 20, SEED, sp)
            env.sync(sp)
            k += 20
    clocks = sampler.stop() if rank == 0 else None
    barrier()

    # the CMA-ES `tell` exchange at the reference controller's size (N = 673 parameters at 32 rays, Controller.cpp:3-8):
    # all-reduce of the weighted mean (N) and the rank-mu sum (N x N), CmaEsSolverTorch.cpp:98-119
    cma_us = None
    if dist is not None:
        buf = torch.zeros(673 * 673 + 673, device="cuda")
        for _ in range(3):
            dist.all_reduce(buf)
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        c0.record(stream)
        for _ in range(20):
            dist.all_reduce(buf)
        c1.record(stream)
        barrier()
        cma_us = 1e3 * c0.elapsed_time(c1) / 20

    # ---- end-to-end arm: HOST buffers through ok_step_host ---------------------------------------
    # as many timed ticks as the device-resident arm; the host action rows repeat after 200 ticks
    e2e_steps = args.steps
    rows = min(e2e_steps, 200)
    thr = ok.pinned_array((max(rows, 3), n), np.float32)
    steer = ok.pinned_array((max(rows, 3), n), np.float32)
    rng = np.random.default_rng(1234 + rank)
    thr[:] = rng.random(thr.shape, dtype=np.float32) * 100.0
    steer[:] = rng.random(steer.shape, dtype=np.float32) * 10.0 - 5.0
    obs = ok.pinned_array((n, N_RAYS), np.float32)
    rew = ok.pinned_array((n,), np.float32)
    done = ok.pinned_array((n,), np.uint8)
    for i in range(3):
        env.step_host(thr[i], steer[i], obs, rew, done, sp)
    barrier()
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    tw = time.perf_counter()
    for i in range(e2e_steps):
        env.step_host(thr[i % rows], steer[i % rows], obs, rew, done, sp)
    e1.record(stream)
    barrier()
    tw = time.perf_counter() - tw
    e2e_ms = max(e0.elapsed_time(e1), 1e3 * tw) / e2e_steps  # host-synchronous path: the wall clock is the honest one
    h2d = 2 * 4 * n
    d2h = n * N_RAYS * 4 + n * 4 + n
    # the same loop with the opt-in, LOSSY 16-bit fixed-point observations (ok_step_host_q16): half the bytes on the link
    # that bounds this path.  Reported next to `e2e`, never as it.
    q16_ms = None
    try:
        obs_q = ok.pinned_array((n, N_RAYS), np.uint16)
        for i in range(3):
            env.step_host(thr[i], steer[i], obs_q, rew, done, sp)
        barrier()
        tq = time.perf_counter()
        for i in range(e2e_steps):
            env.step_host(thr[i % rows], steer[i % rows], obs_q, rew, done, sp)
        barrier()
        q16_ms = 1e3 * (time.perf_counter() - tq) / e2e_steps
    except Exception as ex:  # an experiment build (OK_B200_LIB) without the entry point
        print(f"e2e q16 leg skipped: {ex}", file=sys.stderr)
    # what the host link gives this rank while EVERY rank is moving the same bytes (a bare 8.7 MB device->host transfer
    # per step, nothing else): the ceiling of any end-to-end path on this box
    barrier()
    link = {}
    for pm in ("d2h", "store"):
        try:
            link[pm] = ok.pcie_probe(local, d2h, 40, pm)
        except Exception as ex:
            link[pm] = None
            link["error"] = str(ex)
        barrier()

    # ---- max / min over ranks ----------------------------------------------------------------------
    if dist is not None:
        t = torch.tensor([ms_per_step, e2e_ms, ms_tick, gen_ms, -(link.get("d2h") or 0.0), -(link.get("store") or 0.0)],
                         dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_per_step, e2e_ms, ms_tick, gen_ms = float(t[0]), float(t[1]), float(t[2]), float(t[3])
        link["d2h"], link["store"] = -float(t[4]), -float(t[5])  # the slowest rank's share
        tq = torch.tensor([q16_ms if q16_ms is not None else float("inf")], dtype=torch.float64, device="cuda")
        dist.all_reduce(tq, op=dist.ReduceOp.MAX)
        q16_ms = float(tq[0]) if float(tq[0]) != float("inf") else None

    c5 = None
    if args.config5 or (dist is not None and os.environ.get("OK_BENCH_CONFIG5", "1") != "0"):
        try:
            c5 = config5_leg(ok, torch, dist, rank, world, local, mode, extra)
        except Exception as ex:
            c5 = {"error": str(ex)}

    if rank == 0:
        total_agents = n * world
        value = total_agents / (ms_per_step * 1e-3)
        peak, peak_src = peak_hbm()
        achieved = n * BYTES_PER_AGENT_STEP / (ms_tick * 1e-3) / 1e9  # per GPU, GB/s, the step kernel's own duration
        ev = ncu_evidence() or {}
        issue = None
        if ev.get("warp_instructions_per_launch") and clocks and clocks.get("sm_mhz") and n == N_AGENTS and args.raycast == "beam":
            # the bound that actually binds: warp instructions issued per second against 4 schedulers x SMs x clock.
            # The instruction count is the committed ncu capture's (same command, same workload); the time is this run's.
            sms = torch.cuda.get_device_properties(local).multi_processor_count
            peak_issue = 4.0 * sms * clocks["sm_mhz"] * 1e6
            ach_issue = ev["warp_instructions_per_launch"] / (ms_tick * 1e-3)
            issue = {"achieved": ach_issue, "peak": peak_issue, "unit": "warp-instructions/s", "frac": ach_issue / peak_issue,
                     "warp_instructions_per_launch": ev["warp_instructions_per_launch"],
                     "active_threads_per_instruction": ev.get("active_threads_per_instruction"),
                     "source": ev.get("source")}
        ceiling_ms = None
        if link.get("d2h"):
            ceiling_ms = d2h / (max(link["d2h"], link.get("store") or 0.0) * 1e6)
        line = {
            "metric": "agent_steps_per_sec", "value": value, "unit": "agent-steps/s",
            "ray_casts_per_sec": value * N_RAYS,
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(n, world),
            "impl_config": {"raycast": args.raycast, "grid_cell_px": float(env.cfg.grid_cell), "beam_cell_px": float(env.cfg.beam_cell),
                            "beam_bins": int(env.cfg.beam_bins), "beam_table_bytes": table_bytes, "setup_s": t_build,
                            "schedule": "feedback tiling (ok_balance_schedule, automatic after launches 16 / 64 / 256)", "schedule_settle_ticks": settle,
                            "l2": "flushed between timed ticks (256 MiB memset)" if flush is not None else "not flushed",
                            "crashed_fraction_at_end": crashed_frac, "wall_s_timed_region": t_wall, "numa": numa,
                            "agent_id_base": "rank * agents_per_gpu"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": ev.get("dram_bytes_per_launch"), "peak_source": peak_src,
                         "traffic_source": ev.get("source"),
                         "algorithmic_bytes_per_launch": n * BYTES_PER_AGENT_STEP, "issue": issue,
                         "kernel_ms": ms_tick,
                         "note": ev.get("note", "not HBM bound: warp-issue bound; see profiles/")},
            "e2e": {"value": total_agents / (e2e_ms * 1e-3), "unit": "agent-steps/s", "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms, "steps": e2e_steps,
                    "host_link": {"d2h_copy_GBps_slowest_rank": link.get("d2h"), "mapped_store_GBps_slowest_rank": link.get("store"),
                                  "what": "a bare transfer of d2h_bytes_per_step, all ranks at once (ok_pcie_probe)",
                                  "ceiling_ms_per_step": ceiling_ms,
                                  "e2e_over_ceiling": (e2e_ms / ceiling_ms) if ceiling_ms else None},
                    "q16_opt_in": None if q16_ms is None else {
                        "value": total_agents / (q16_ms * 1e-3), "ms_per_step": q16_ms,
                        "d2h_bytes_per_step": n * N_RAYS * 2 + n * 4 + n,
                        "what": "ok_step_host_q16: observations as 16-bit fixed point, rn(obs * 65535) -- LOSSY (<= 7.7e-6 of the "
                                "sensor range), opt-in, not the headline"}},
            "gpu_launches": int(launches), "clocks": clocks,
        }
        if dist is not None:
            line["generation"] = {
                "every_ticks": gen_every, "exchanges_timed": len(gens), "collective_us": 1e3 * gen_ms,
                "allgather_us": 1e3 * gather_ms, "ranking_sort_us": 1e3 * (gen_ms - gather_ms),
                "what": "NCCL all-gather of f32 fitness[agents x ranks] + stable global ranking (sort), on the step stream, inside the timed region",
                "bytes_gathered_per_rank": 4 * n * world, "ms_per_tick_without": ms_tick,
                "value_without_collective": total_agents / (ms_tick * 1e-3),
                "cmaes_tell_allreduce_us": cma_us, "cmaes_tell_allreduce_bytes": 4 * (673 * 673 + 673)}
            line["shard_parity"] = shard_parity
            line["shard_parity_what"] = (f"rank 0 replayed agents {n}..{n + min(1024, n) - 1} (rank 1's first) alone for {parity_ticks} ticks: "
                                         f"{len(PARITY_BUFS)} buffers bit-compared")
        if c5 is not None:
            line["config5"] = c5
        if not args.no_cpu:
            if world == 1:
                try:
                    line["ref_cuda_kernel"] = ref_cuda_kernel_baseline(ok)
                except Exception as ex:
                    line["ref_cuda_kernel"] = {"error": str(ex)}
            try:
                _, _, info = cpu_reference_run(steps=10, warmup=2, budget_s=20.0)
                line["cpu_baseline"] = info
            except Exception as ex:  # the bench line must still print
                line["cpu_baseline"] = {"value": None, "unit": "agent-steps/s", "cores": None, "kind": "port",
                                        "sample": f"failed: {ex}"}
        emit(line)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def config5_leg(ok, torch, dist, rank, world, local, mode, extra, n=1 << 20, ticks=40, generations=3):
    """BASELINE configs[4]: a CMA-ES population of 1,048,576 candidates PER GPU (8 M over 8 GPUs), every candidate an
    agent; per generation `ticks` ticks of the step kernel, then the NCCL fitness all-gather + global ranking and the
    N x N `tell` all-reduce.  Short (a few seconds): it reports the shape's tick time and the exchange's cost."""
    from openkitchen_b200 import dist as okdist

    env = ok.Env(device=local, movement_mode=ok.MOVE_VELOCITY, reward_mode=ok.REWARD_CMAES_PROGRESS, auto_reset=1,
                 raycast_mode=mode, agent_id_base=rank * n, **extra)
    build_workload(ok, env, n, id_base=rank * n, period=n)
    stream = torch.cuda.current_stream()
    sp = stream.cuda_stream
    fit = torch.from_dlpack(ok.dlpack.DeviceBuffer(env, "fitness"))
    buf = torch.zeros(673 * 673 + 673, device="cuda")
    env.launch_steps_random(0, 5, SEED, sp)
    okdist.global_ranking(fit, n * world)
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3 * generations + 1)]
    ev[0].record(stream)
    for g in range(generations):
        env.launch_steps_random(5 + g * ticks, ticks, SEED, sp)
        ev[3 * g + 1].record(stream)
        okdist.global_ranking(fit, n * world)
        ev[3 * g + 2].record(stream)
        if dist is not None:
            dist.all_reduce(buf)
        ev[3 * g + 3].record(stream)
    torch.cuda.synchronize()
    tick_ms = sum(ev[3 * g].elapsed_time(ev[3 * g + 1]) for g in range(generations)) / (generations * ticks)
    rank_ms = sum(ev[3 * g + 1].elapsed_time(ev[3 * g + 2]) for g in range(generations)) / generations
    tell_ms = sum(ev[3 * g + 2].elapsed_time(ev[3 * g + 3]) for g in range(generations)) / generations
    total_ms = ev[0].elapsed_time(ev[-1])
    t = torch.tensor([tick_ms, rank_ms, tell_ms, total_ms], dtype=torch.float64, device="cuda")
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    tick_ms, rank_ms, tell_ms, total_ms = (float(v) for v in t)
    env.close()
    return {"workload": f"C5 shape: {n} agents per GPU x {world} GPUs x {N_RAYS} rays, {ticks} ticks per generation, {generations} generations",
            "agents_total": n * world, "ms_per_tick": tick_ms, "agent_steps_per_sec_ticks_only": n * world / (tick_ms * 1e-3),
            "fitness_allgather_rank_ms": rank_ms, "fitness_bytes": 4 * n * world, "tell_allreduce_ms": tell_ms,
            "agent_steps_per_sec_with_exchange": n * world * ticks * generations / (total_ms * 1e-3),
            "l2": "not flushed (state of 1M agents = 1.4 GB per tick, far larger than L2)"}


def emit(line):
    """the ONE JSON line of the contract, on the process's real stdout"""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1

if __name__ == "__main__":
    # Libraries write to file descriptor 1 behind Python's back (NCCL prints "NCCL version ..." there when NCCL_DEBUG is set):
    # keep the real stdout for the one JSON line and point fd 1 at stderr for everything else.
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    main()

"""Mints tests/golden/sizing_plans.json: the kernel shape and beam tiling ok_alloc_agents chooses for named populations,
as launch_stats() and debug_tiles() report them right after alloc_agents, with the device facts they were chosen from.
tests/test_schedule_cpu.py replays the same inputs through the sizing functions of ok_schedule.cpp on the CPU.

usage (on a GPU host): python tools/make_golden_sizing.py OUT.json   (OK_B200_LIB selects another build of the library)"""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import openkitchen_b200 as ok  # noqa: E402

BENCH = dict(n=65536, rays=32)  # bench.py's population
# every shape runs over all 23 packed tracks, track_id = i * 23 // n (contiguous per track, as bench.py)
SHAPES = {
    "bench-beam": dict(BENCH, raycast="beam", knobs={}),
    "bench-grid": dict(BENCH, raycast="grid", knobs={}),
    "bench-waves3": dict(BENCH, raycast="beam", knobs={"OK_BEAM_WAVES": "3"}),
    "bench-tail4": dict(BENCH, raycast="beam", knobs={"OK_BEAM_TAIL": "4"}),
    "bench-batch96": dict(BENCH, raycast="beam", knobs={"OK_BEAM_BATCH_AGENTS": "96"}),
    "bench-flushers8": dict(BENCH, raycast="beam", knobs={"OK_E2E_FLUSHERS": "8"}),
    "bench-unstaged": dict(BENCH, raycast="beam", knobs={"OK_BEAM_KERNEL": "unstaged"}),
    "300-staged": dict(n=300, rays=32, raycast="beam", knobs={"OK_BEAM_KERNEL": "staged"}),
    "300-unstaged": dict(n=300, rays=32, raycast="beam", knobs={"OK_BEAM_KERNEL": "unstaged"}),
    "4096x5": dict(n=4096, rays=5, raycast="beam", knobs={}),
    "one-agent": dict(n=1, rays=32, raycast="beam", knobs={}),
}
MODES = {"beam": ok.RAYCAST_BEAM, "grid": ok.RAYCAST_GRID}


def main(out_path):
    names = ok.track_names()
    host = ok.Env(device=-1)
    for nm in names:
        host.add_named_track(nm)
    props = torch.cuda.get_device_properties(0)
    facts = {"gpu": props.name, "num_sms": props.multi_processor_count, "smem_optin": props.shared_memory_per_block_optin,
             "max_blob": max(host.track_info(t).blob_bytes for t in range(len(names)))}
    plans = {}
    for name, s in SHAPES.items():
        for k, v in s["knobs"].items():
            os.environ[k] = v
        try:
            env = ok.Env(device=0, raycast_mode=MODES[s["raycast"]])
            for nm in names:
                env.add_named_track(nm)
            tid = (np.arange(s["n"]) * len(names) // s["n"]).astype(np.int32)
            env.alloc_agents(s["n"], ok.ray_fan(s["rays"]), tid)
            st = env.launch_stats()
            plans[name] = dict(s, grid=st.grid_blocks, block=st.block_threads, smem=st.smem_bytes, tiles=st.tiles,
                               debug_tiles=np.asarray(env.debug_tiles()).reshape(-1, 3).tolist())
            env.close()
        finally:
            for k in s["knobs"]:
                del os.environ[k]
    with open(out_path, "w") as f:  # one plan per line
        f.write('{"device": %s,\n "plans": {\n' % json.dumps(facts))
        f.write(",\n".join("  %s: %s" % (json.dumps(k), json.dumps(v, separators=(",", ":"))) for k, v in plans.items()))
        f.write("\n }\n}\n")
    print(json.dumps({k: {q: v[q] for q in ("grid", "block", "smem", "tiles")} for k, v in plans.items()}))


if __name__ == "__main__":
    main(sys.argv[1])

#!/usr/bin/env python
"""Pack the 23 TUMFTM racetrack-database centre lines the reference ships (tracks/*.csv) into one
binary file so that the benchmark / tests have BASELINE.json's tracks without a checkout of the
original project.

The pack stores the four raw CSV columns (x_m, y_m, w_tr_right_m, w_tr_left_m) as binary32 exactly
as std::stof (strtof) parses them -- the parse goes through the oracle's strtof-based loader's
twin below and is cross-checked against it in tests/test_tracks.py when the CSVs are present.

Usage:  python tools/make_track_pack.py [$OPENKITCHEN_REF/tracks] [openkitchen_b200/data/tracks_f32.npz]
"""
import ctypes
import glob
import os
import sys

import numpy as np

libc = ctypes.CDLL(None)
libc.strtof.restype = ctypes.c_float
libc.strtof.argtypes = [ctypes.c_char_p, ctypes.c_void_p]


def parse_csv(path):
    cols = [[], [], [], []]
    with open(path, "rb") as f:
        f.readline()  # RaceTrack.cpp:136-137 skips the first line
        for line in f:
            toks = line.strip().split(b",")
            if len(toks) < 4:
                continue
            for c in range(4):
                cols[c].append(libc.strtof(toks[c], None))
    return [np.asarray(c, dtype=np.float32) for c in cols]


def main():
    src = sys.argv[1] if len(sys.argv) > 1 else os.path.join(os.environ.get("OPENKITCHEN_REF", "."), "tracks")
    dst = sys.argv[2] if len(sys.argv) > 2 else os.path.join(os.path.dirname(__file__), "..", "openkitchen_b200", "data", "tracks_f32.npz")
    out = {}
    names = []
    for p in sorted(glob.glob(os.path.join(src, "*.csv"))):
        name = os.path.splitext(os.path.basename(p))[0]
        x, y, wr, wl = parse_csv(p)
        out[name] = np.stack([x, y, wr, wl], axis=0)
        names.append(name)
    out["__names__"] = np.array(names)
    np.savez_compressed(dst, **out)
    print(f"packed {len(names)} tracks, {sum(out[n].shape[1] for n in names)} points -> {dst} ({os.path.getsize(dst)} bytes)")


if __name__ == "__main__":
    main()

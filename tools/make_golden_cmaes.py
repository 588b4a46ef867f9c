#!/usr/bin/env python
"""Mints tests/golden/cmaes_ref.npz from the reference's OWN CMA-ES solver and controller
(oracle/_ref/libcmaes_ref.so = CmaEsSolverTorch.cpp + Controller.cpp compiled unchanged, oracle/Makefile).
Needs a checkout of the original project:  OPENKITCHEN_REF=<checkout> make -C oracle && python tools/make_golden_cmaes.py"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle.cmaes_oracle import CmaEsReference, have_ref, reference_controller_forward  # noqa: E402

N, LAM, GENS = 24, 20, 8  # kPopulationSize 20 (main_torch.cpp:12)


def fitness(x):
    return (-((x - 0.3) ** 2).sum(-1) + 0.1 * np.sin(5 * x).sum(-1)).astype(np.float32)


def main():
    if not have_ref():
        raise SystemExit("oracle/_ref/libcmaes_ref.so missing: make -C oracle")
    out = {}
    ref = CmaEsReference(N, LAM)
    for k, v in ref.state().items():
        out[f"init_{k}"] = v
    for g in range(GENS):
        torch.manual_seed(1000 + g)
        x = ref.sample().numpy()
        f = fitness(x)
        ref.tell(x, f)
        out[f"g{g}_x"], out[f"g{g}_fit"] = x, f
        for k, v in ref.state().items():
            out[f"g{g}_{k}"] = v
    rng = np.random.default_rng(11)
    for rays in (5, 32, 128):  # QAgent fan, the bench fan, main_torch.cpp:26
        p = 16 * rays + 16 + 136 + 9
        flat = (rng.standard_normal((6, p)) * 0.4).astype(np.float32)
        obs = rng.random((6, rays)).astype(np.float32)
        out[f"ctrl{rays}_flat"], out[f"ctrl{rays}_obs"] = flat, obs
        out[f"ctrl{rays}_out"] = reference_controller_forward(flat, obs, rays)
    path = os.path.join(ROOT, "tests", "golden", "cmaes_ref.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()

"""Lap accounting (OkLaps, include/openkitchen_b200.h) over the parity oracles (TEST INFRASTRUCTURE ONLY).

The oracles of oracle/ are left as they are; this module adds the accounting around them.  The seven per-agent arrays live
here in numpy.  A restart takes the nearest index a reset leaves in the oracle's prev_idx buffer.  A tick with accounting on
first resets, through ``Oracle.reset`` (or the drawn reset of tests/reset_draws_oracle.py), every agent the tick's
auto-reset takes: the crashed ones and the completed ones, at the stride point.  The oracle's own auto-reset then finds no
crashed agent.  After ``Oracle.step`` it applies rule 2 to the agents that moved, with n from ``Oracle.nearest_index``,
and writes n to the nearest_idx buffer and crashed || completed to the done buffer, as the laps kernels do.
"""
from __future__ import annotations

import numpy as np

from oracle.api import Oracle

FIELDS = {"lap_idx": np.int32, "progress": np.int32, "laps": np.int32, "ticks": np.uint32, "lap_start": np.uint32,
          "last_lap": np.uint32, "completed": np.uint8}
_PROGRESS_MODES = (1, 2, 6, 7)  # the reward modes whose oracle tick already searches the nearest index


def _i32(x):
    """two's-complement wrap of int64 values to int32"""
    return ((np.asarray(x, dtype=np.int64) + 2**31) % 2**32 - 2**31).astype(np.int32)


def lap_rule(s: dict, n, P, target: int, moved) -> dict:
    """Rule 2 of the header, vectorised: the state dict `s` (FIELDS) after a tick in which the agents with moved != 0 went
    to nearest index n on tracks of P points.  Returns a new dict; agents that did not move keep their state."""
    moved = np.asarray(moved, dtype=bool)
    n = np.asarray(n, dtype=np.int64)
    P = np.broadcast_to(np.asarray(P, dtype=np.int64), moved.shape)
    d = _i32(n - s["lap_idx"].astype(np.int64)).astype(np.int64)
    d = np.where(2 * d > P, d - P, np.where(2 * d <= -P, d + P, d))
    progress = _i32(s["progress"].astype(np.int64) + d)
    ticks = (s["ticks"].astype(np.uint64) + 1).astype(np.uint32)
    lap = progress.astype(np.int64) >= (s["laps"].astype(np.int64) + 1) * P
    laps = np.where(lap, _i32(s["laps"].astype(np.int64) + 1), s["laps"])
    last_lap = np.where(lap, ticks - s["lap_start"], s["last_lap"]).astype(np.uint32)
    lap_start = np.where(lap, ticks, s["lap_start"]).astype(np.uint32)
    completed = np.where((target > 0) & (laps >= target), np.uint8(1), s["completed"]).astype(np.uint8)
    new = {"lap_idx": n.astype(np.int32), "progress": progress, "laps": laps, "ticks": ticks, "lap_start": lap_start,
           "last_lap": last_lap, "completed": completed}
    return {f: np.where(moved, new[f], s[f]).astype(dt) for f, dt in FIELDS.items()}


class Laps:
    """The lap accounting of one oracle (after its alloc_agents and its first reset), optionally with the reset draws of a
    ``DrawnResets`` of the same oracle: ``set`` (ok_set_laps), ``reset`` (an explicit reset with restart), ``step`` (a
    tick) and the arrays ``s``."""

    def __init__(self, ora: Oracle, drawn=None):
        self.ora, self.drawn = ora, drawn
        self.n_points = np.array([ora.track_points(int(t)) for t in ora.buffer("track_id")], dtype=np.int64)
        self.s = {f: np.zeros(ora.n, dtype=dt) for f, dt in FIELDS.items()}
        self.restart(np.arange(ora.n))  # what the initial reset of ok_alloc_agents leaves
        self.enabled, self.target = False, 0

    def _nearest(self, idx):
        tid, x, y = self.ora.buffer("track_id"), self.ora.buffer("pos_x"), self.ora.buffer("pos_y")
        return np.array([self.ora.nearest_index(int(tid[a]), float(x[a]), float(y[a])) for a in idx], dtype=np.int32)

    def restart(self, idx, near=None):
        """rule 1 for agents idx at the nearest index of their pose (default: prev_idx, which a reset has just set)"""
        idx = np.asarray(idx, dtype=np.int64)
        for f in FIELDS:
            self.s[f][idx] = 0
        self.s["lap_idx"][idx] = self.ora.buffer("prev_idx")[idx] if near is None else near

    def set(self, enabled: bool, target: int = 0):
        if enabled and not self.enabled:
            every = np.arange(self.ora.n)
            self.restart(every, self._nearest(every))
        self.enabled, self.target = bool(enabled), int(target)

    def reset(self, agent_idx, pt_idx, lane_alpha=None, heading_off=None):
        self.ora.reset(agent_idx, pt_idx, lane_alpha, heading_off)
        self.restart(np.arange(self.ora.n) if agent_idx is None else agent_idx)

    def step(self):
        """Oracle.step (through the DrawnResets, if any) with the accounting of the header"""
        ora = self.ora
        if not self.enabled:
            (self.drawn.step if self.drawn is not None else ora.step)()
            return
        if ora.cfg.auto_reset:
            idx = np.flatnonzero((ora.buffer("crashed") != 0) | (self.s["completed"] != 0))
            stride = ((ora.buffer("reset_pt")[idx].astype(np.int64) + ora.cfg.auto_reset_stride) % self.n_points[idx]).astype(np.int32)
            if self.drawn is not None and self.drawn.flags:
                self.drawn._reset(idx, stride)
            elif idx.size:
                ora.reset(idx, stride)
            self.restart(idx)
        moved = ora.buffer("crashed") == 0
        ora.step()
        every = np.arange(ora.n)
        if ora.cfg.reward_mode in _PROGRESS_MODES:
            n = ora.buffer("nearest_idx").copy()
        else:
            n = self._nearest(every)
            ora.buffer("nearest_idx")[:] = n
        self.s = lap_rule(self.s, n, self.n_points, self.target, moved)
        ora.buffer("done")[:] = (ora.buffer("crashed") != 0) | (self.s["completed"] != 0)

"""Reset draws (OkResetDraws, include/openkitchen_b200.h) over the parity oracles (TEST INFRASTRUCTURE ONLY).

The oracles of oracle/ are left as they are; this module adds the draws around them.  A drawn reset is
``Oracle.reset`` (the oracle's Environment::resetAgent with explicit draws) fed the (pt, alpha, offset) of the header's
definition, restated here in numpy (``draw``), with the per-agent counters k kept here.  The drawn auto-reset of a tick is
that reset of every crashed agent just before ``Oracle.step``: the oracle's own auto-reset then finds no crashed agent,
and the tick runs the reset agents with the zero action the reset wrote, as the stride auto-reset does.
"""
from __future__ import annotations

import numpy as np

from oracle.api import Oracle

POINT, LANE, HEADING = 1, 2, 4
RESET_KEY = 0x525354  # "RST": the second key word of the reset stream
STARTING_IDX = 3      # RaceTrack::kStartingIdx: an explicit reset's point without OK_RESET_DRAW_POINT
_M32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 (Salmon et al., SC'11) on arrays of 32-bit words, vectorised; the four output words as uint64 arrays.
    Pinned to the oracle's oko_philox4x32_10 by tests/test_reset_draws_cpu.py."""
    c = [np.asarray(x, dtype=np.uint64) & _M32 for x in (c0, c1, c2, c3)]
    k0, k1 = np.asarray(k0, dtype=np.uint64) & _M32, np.asarray(k1, dtype=np.uint64) & _M32
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c[0]
        p1 = np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & _M32, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & _M32]
        k0 = (k0 + np.uint64(0x9E3779B9)) & _M32
        k1 = (k1 + np.uint64(0xBB67AE85)) & _M32
    return c


def draw(seed, flags, ids, k, n_points, pt_otherwise):
    """The header's definition: (pt i32, alpha f32, heading offset f32) of the drawn resets of agents with global ids `ids`
    at counters `k`; n_points and pt_otherwise (the point without OK_RESET_DRAW_POINT) per agent or scalar.  alpha is
    meaningful only with OK_RESET_DRAW_LANE."""
    ids, k = np.asarray(ids, dtype=np.uint64), np.asarray(k, dtype=np.uint64)
    o = philox4x32_10(ids & _M32, ids >> np.uint64(32), k, 0, seed, RESET_KEY)

    def below(w, m):  # U(o, m) = (o * m) >> 32
        return ((w * np.asarray(m, dtype=np.uint64)) >> np.uint64(32)).astype(np.int64)

    if flags & POINT:
        pt = below(o[0], n_points).astype(np.int32)
    else:
        pt = np.broadcast_to(np.asarray(pt_otherwise, dtype=np.int32), ids.shape).astype(np.int32)
    alpha = ((np.float32(10) + below(o[1], 81).astype(np.float32)) / np.float32(100)).astype(np.float32)
    if flags & HEADING:
        mag = (45 + below(o[2], 46)).astype(np.float32)
        off = np.where(k & np.uint64(1), mag, -mag).astype(np.float32)
    else:
        off = np.zeros(ids.shape, dtype=np.float32)
    return pt, alpha, off


class DrawnResets:
    """The reset draws of one oracle (``"port"`` or ``"reference"``, after its alloc_agents): ``set``, ``reset`` (the
    explicit drawn reset), ``step`` (a tick whose auto-reset draws when the oracle's auto_reset is on) and the counters
    ``k``."""

    def __init__(self, ora: Oracle, seed: int = 0, flags: int = 0):
        self.ora = ora
        self.k = np.zeros(ora.n, dtype=np.uint32)
        tid = ora.buffer("track_id")
        self.n_points = np.array([ora.track_points(int(t)) for t in tid], dtype=np.int64)
        self.set(seed, flags)

    def set(self, seed: int, flags: int):
        self.seed, self.flags = int(seed) & 0xFFFFFFFF, int(flags)

    def _reset(self, idx, pt_otherwise):
        idx = np.asarray(idx, dtype=np.int64)
        if idx.size == 0:
            return
        ids = np.uint64(self.ora.cfg.agent_id_base) + idx.astype(np.uint64)
        pt, alpha, off = draw(self.seed, self.flags, ids, self.k[idx], self.n_points[idx], pt_otherwise)
        self.ora.reset(idx, pt, alpha if self.flags & LANE else None, off)
        self.k[idx] += np.uint32(1)

    def reset(self, agent_idx=None, mask=None):
        """drawn reset of agent_idx | the agents where mask != 0 | all agents"""
        if agent_idx is not None:
            idx = np.asarray(agent_idx, dtype=np.int64)
        elif mask is not None:
            idx = np.flatnonzero(np.asarray(mask))
        else:
            idx = np.arange(self.ora.n)
        self._reset(idx, np.minimum(STARTING_IDX, self.n_points[idx] - 1))

    def step(self):
        """Oracle.step with the drawn auto-reset (draws on and the oracle's auto_reset set), else Oracle.step as it is"""
        if self.flags and self.ora.cfg.auto_reset:
            idx = np.flatnonzero(self.ora.buffer("crashed"))
            stride = (self.ora.buffer("reset_pt")[idx].astype(np.int64) + self.ora.cfg.auto_reset_stride) % self.n_points[idx]
            self._reset(idx, stride)
        self.ora.step()

"""Races (OkRaces, include/openkitchen_b200.h) over the port oracle (TEST INFRASTRUCTURE ONLY).

The oracles of oracle/ are left as they are; this module restates the race pass on the oracle's buffers in numpy float32,
one agent at a time, after each ``Oracle.step`` / ``Oracle.cast_rays``.  numpy's float32 operations are single correctly
rounded operations (no contraction), and its float32 sqrt is correctly rounded, so the restatement follows the header's
order of operations bit for bit.  The ray directions come from ``Oracle.sincosf`` (the restatement of the device
sincosf).  The pass's own outputs, ``hit_car`` and ``contact``, live here.
"""
from __future__ import annotations

import math

import numpy as np

from oracle.api import Oracle

SENSE, CONTACT = 1, 2
K_DEG2RAD = np.float32(0.0174532924)
F32 = np.float32


class Races:
    """The race pass of one oracle: ``apply`` after every tick that casts rays; ``hit_car`` i32[N, R] and ``contact`` u8[N]
    as the pass leaves them.  ``fan`` is the oracle's ray fan (degrees)."""

    def __init__(self, ora: Oracle, fan, group: int, radius: float, flags: int = SENSE | CONTACT):
        self.ora, self.fan = ora, np.asarray(fan, dtype=np.float32)
        self.group, self.radius, self.flags = int(group), F32(radius), int(flags)
        self.hit_car = np.full((ora.n, ora.rays), -1, dtype=np.int32)
        self.contact = np.zeros(ora.n, dtype=np.uint8)
        # totals over every pass, what a test really exercised: rays that hit a car (and of those, from inside the body),
        # agents crashed by contact and by what the lidar saw
        self.car_hits = self.inside_hits = self.contact_crashes = self.sense_crashes = 0

    def opponents(self, i: int) -> np.ndarray:
        """the opponents of agent i, ascending: same race, same track, not i"""
        tid = self.ora.buffer("track_id")
        lo = i // self.group * self.group
        js = np.arange(lo, min(lo + self.group, self.ora.n))
        return js[(tid[js] == tid[i]) & (js != i)]

    def rays(self, i: int):
        """the lidar origin (ox, oy), (rc, rs) of the heading and the rays' directions (dx, dy) of agent i, as the tick
        computed them"""
        ora, cfg = self.ora, self.ora.cfg
        x, y, rot = ora.buffer("pos_x")[i], ora.buffer("pos_y")[i], ora.buffer("rot")[i]
        rs, rc = (F32(v) for v in ora.sincosf(float(K_DEG2RAD * rot)))
        off = F32(cfg.sensor_offset)
        ox, oy = x + off * rc, y + off * rs
        dirs = np.array([ora.sincosf(float(a)) for a in K_DEG2RAD * (rot + self.fan)], dtype=np.float32)
        return ox, oy, rc, rs, dirs[:, 1], dirs[:, 0]

    def car_t(self, ox, oy, dx, dy, xj, yj) -> np.ndarray:
        """t[r, k] of ray r against body k (inf = missed or beyond sensor_range), the header's expression"""
        rr = self.radius * self.radius
        wx, wy = xj - ox, yj - oy
        b = wx[None, :] * dx[:, None] + wy[None, :] * dy[:, None]
        c = (wx * wx + wy * wy) - rr
        q = b * b - c[None, :]
        t = np.where(c[None, :] <= 0, F32(0), np.where((b > 0) & (q >= 0), np.fmax(b - np.sqrt(q), F32(0)), F32(np.inf)))
        return np.where(t <= F32(self.ora.cfg.sensor_range), t, F32(np.inf)).astype(np.float32)

    def apply(self):
        ora, cfg = self.ora, self.ora.cfg
        x, y = ora.buffer("pos_x"), ora.buffer("pos_y")
        crashed, done = ora.buffer("crashed"), ora.buffer("done")
        habs, hrel, obs = ora.buffer("hit_abs"), ora.buffer("hit_rel"), ora.buffer("obs")
        ht, hseg, md2 = ora.buffer("hit_t"), ora.buffer("hit_seg"), ora.buffer("min_dist2")
        rng_, cd2 = F32(cfg.sensor_range), F32(cfg.collision_dist2)
        live = np.flatnonzero(crashed == 0)  # the crash flags as the pass starts
        self.contact[:] = 0
        with np.errstate(invalid="ignore", over="ignore"):
            for i in live:
                opp = self.opponents(int(i))
                crash = False
                if self.flags & CONTACT and opp.size:
                    ddx, ddy = x[i] - x[opp], y[i] - y[opp]
                    d = self.radius + self.radius
                    if np.any(ddx * ddx + ddy * ddy < d * d):
                        crash = True
                        self.contact_crashes += 1
                if self.flags & SENSE:
                    self.hit_car[i] = -1
                    if opp.size:
                        ox, oy, rc, rs, dx, dy = self.rays(int(i))
                        t = self.car_t(ox, oy, dx, dy, x[opp], y[opp])
                        k = np.argmin(t, axis=1)  # the first minimum: the lowest j among ties
                        bt = t[np.arange(t.shape[0]), k]
                        rep = np.isfinite(bt) & (bt < ht[i])
                        for r in np.flatnonzero(rep):
                            tr = bt[r]
                            hx, hy = ox + tr * dx[r], oy + tr * dy[r]
                            xt, yt = hx - ox, hy - oy
                            rx, ry = xt * rc - yt * rs, xt * rs + yt * rc
                            habs[i, r] = (hx, hy)
                            hrel[i, r] = (rx, ry)
                            obs[i, r] = np.sqrt(rx * rx + ry * ry) / rng_
                            ht[i, r], hseg[i, r] = tr, -1
                            self.hit_car[i, r] = opp[k[r]]
                        if rep.any():
                            self.car_hits += int(rep.sum())
                            self.inside_hits += int(np.sum(bt[rep] == 0))
                            sq = hrel[i, :, 0] * hrel[i, :, 0] + hrel[i, :, 1] * hrel[i, :, 1]
                            m = rng_ * rng_  # `if (sq < min) min = sq` over the rays: NaN never wins
                            for v in sq:
                                if v < m:
                                    m = v
                            md2[i] = m
                            if m < cd2:
                                crash = True
                                self.sense_crashes += 1
                if crash:
                    crashed[i], done[i], self.contact[i] = 1, 1, 1


def pack_races(x, y, rot, tid, group: int, rng, spacing=(1.0, 5.0, 8.5, 12.0, 30.0, 90.0, 250.0)):
    """poses (new float32 arrays) with the cars of each race and track lined up along its first car's heading at random
    spacings (overlapping, in the lidar's crash band, in range and out of range), a little off the line, at headings
    within 40 degrees of it or reversed"""
    x, y, rot = (np.array(v, dtype=np.float32) for v in (x, y, rot))
    n = len(x)
    for lo in range(0, n, group):
        members = np.arange(lo, min(lo + group, n))
        for t in np.unique(tid[members]):
            same = members[tid[members] == t]
            if same.size < 2:
                continue
            lead = same[0]
            a = math.radians(float(rot[lead]))
            d = np.cumsum(rng.choice(spacing, same.size - 1))
            side = rng.uniform(-6.0, 6.0, same.size - 1)
            x[same[1:]] = (x[lead] + d * math.cos(a) - side * math.sin(a)).astype(np.float32)
            y[same[1:]] = (y[lead] + d * math.sin(a) + side * math.cos(a)).astype(np.float32)
            turn = rng.uniform(-40, 40, same.size - 1) + rng.choice([0, 180], same.size - 1)
            rot[same[1:]] = (rot[lead] + turn).astype(np.float32)
    return x, y, rot

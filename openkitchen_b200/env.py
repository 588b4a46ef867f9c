"""Thin object wrapper over the C ABI: one :class:`Env` per GPU.

This layer holds no algorithm: every method is one call into ``libopenkitchen_b200.so``.  numpy
arrays cross the boundary as HOST buffers (``*_host`` / read / write entry points); device pointers
are exposed as integers for the torch / DLPack layer in :mod:`openkitchen_b200.batch_env`.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import _capi
from ._capi import BUF, OkConfig, OkLaunchStats, OkPopulationCounters, OkTrackInfo, check

_NP_DTYPES = {_capi.DTYPE_F32: np.float32, _capi.DTYPE_I32: np.int32, _capi.DTYPE_U32: np.uint32, _capi.DTYPE_U8: np.uint8}
_DATA = os.path.join(os.path.dirname(os.path.abspath(__file__)), "data", "tracks_f32.npz")


def _vp(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def track_names():
    """Names of the 23 racetrack-database tracks packed in data/tracks_f32.npz (sorted)."""
    with np.load(_DATA) as z:
        return [str(n) for n in z["__names__"]]


def track_columns(name: str):
    """The four raw CSV columns (x_m, y_m, w_tr_right_m, w_tr_left_m) of a packed track, binary32."""
    with np.load(_DATA) as z:
        a = z[name]
    return a[0].copy(), a[1].copy(), a[2].copy(), a[3].copy()


def write_track_csv(name: str, path: str):
    """Re-emit a packed track in the reference's CSV format (%.9g round-trips binary32 through stof)."""
    x, y, wr, wl = track_columns(name)
    with open(path, "w") as f:
        f.write("# x_m,y_m,w_tr_right_m,w_tr_left_m\n")
        for i in range(len(x)):
            f.write("%.9g,%.9g,%.9g,%.9g\n" % (x[i], y[i], wr[i], wl[i]))


def release_caches() -> None:
    """drop the process-wide beam-table caches (tables in use by live envs stay alive until those envs are closed)"""
    _capi.load().ok_release_caches()


def ray_fan(n_rays: int) -> np.ndarray:
    """Evenly spaced fan -70..70 deg in binary32: the generator of main_torch.cpp:26-34."""
    if n_rays == 1:
        return np.zeros(1, dtype=np.float32)
    i = np.arange(n_rays, dtype=np.int32).astype(np.float32)
    return (np.float32(-70.0) + (i * np.float32(140.0)) / np.float32(n_rays - 1)).astype(np.float32)


# the outputs of a lidar query, by their BatchEnv names: (OkLidarQuery field, numpy dtype, shape for (poses, rays))
LIDAR_OUTPUTS = {
    "obs": ("obs", np.float32, lambda n, r: (n, r)),
    "hits": ("hit_rel", np.float32, lambda n, r: (n, r, 2)),
    "hit_points": ("hit_abs", np.float32, lambda n, r: (n, r, 2)),
    "hit_seg": ("hit_seg", np.int32, lambda n, r: (n, r)),
    "hit_t": ("hit_t", np.float32, lambda n, r: (n, r)),
    "min_dist2": ("min_dist2", np.float32, lambda n, r: (n,)),
    "crashed": ("crashed", np.uint8, lambda n, r: (n,)),
}


def _pose_arrays(x, y, rot, track_id=None):
    """x, y, rot as contiguous binary32 vectors of one length (and track_id of that length); raises ValueError otherwise"""
    x, y, rot = (np.ascontiguousarray(a, dtype=np.float32) for a in (x, y, rot))
    if x.ndim != 1 or x.shape != y.shape or x.shape != rot.shape:
        raise ValueError("x, y and rot must be 1-d arrays of one length")
    if track_id is not None and np.shape(track_id) != x.shape:
        raise ValueError("track_id must have one entry per pose")
    return x, y, rot


def _bev_shape(height, width, scale, ahead):
    """the image arguments of a bird's-eye-view query, checked as the library checks them; raises ValueError otherwise"""
    height, width = int(height), int(width)
    with np.errstate(over="ignore"):  # the library sees binary32: 1e39 is inf there
        scale, ahead = np.float32(scale), np.float32(ahead)
    if not (1 <= height <= 1024 and 1 <= width <= 1024):
        raise ValueError("height and width must be in 1..1024")
    if not (np.isfinite(scale) and scale > 0):
        raise ValueError("scale must be finite and > 0")
    if not np.isfinite(ahead):
        raise ValueError("ahead must be finite")
    scale, ahead = float(scale), float(ahead)
    return height, width, scale, ahead


class Env:
    """Owns one ``OkEnv``.  ``device=-1`` builds a host-only env (tracks can be built and inspected)."""

    def __init__(self, device: int = 0, **cfg):
        self.lib = _capi.load()
        c = OkConfig()
        self.lib.ok_config_default(C.byref(c))
        c.device = device
        for k, v in cfg.items():
            if not hasattr(c, k):
                raise AttributeError(f"OkConfig has no field {k}")
            setattr(c, k, v)
        self.cfg = c
        h = C.c_void_p()
        check(self.lib.ok_create(C.byref(c), C.byref(h)))
        self.h = h
        self.n = 0
        self.rays = 0

    # ---- lifetime -----------------------------------------------------------------------
    def close(self):
        """Destroys the OkEnv -- unless DLPack tensors exported from it are still alive: device memory a consumer can
        still touch is never freed under it; the env is then destroyed when its last export is released."""
        if not getattr(self, "h", None):
            return
        from . import dlpack

        if dlpack.live_exports(self) > 0:
            self._close_pending = True
            return
        self._destroy_now()

    def _destroy_now(self):
        if getattr(self, "h", None):
            self.lib.ok_destroy(self.h)
            self.h = None
        self._close_pending = False

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def update_config(self, **cfg):
        """change per-tick constants of the live env (movement_mode, reward_mode, auto_reset, ...)"""
        for k, v in cfg.items():
            if not hasattr(self.cfg, k) or k in ("device", "grid_cell", "beam_cell", "beam_bins"):
                raise AttributeError(f"cannot update {k}")
            setattr(self.cfg, k, v)
        check(self.lib.ok_update_config(self.h, C.byref(self.cfg)))

    # ---- tracks -------------------------------------------------------------------------
    def add_track(self, cols) -> int:
        x, y, wr, wl = (np.ascontiguousarray(c, dtype=np.float32) for c in cols)
        tid = C.c_int32(-1)
        check(self.lib.ok_add_track(self.h, _vp(x), _vp(y), _vp(wr), _vp(wl), len(x), C.byref(tid)))
        return tid.value

    def add_named_track(self, name: str) -> int:
        return self.add_track(track_columns(name))

    def load_track_csv(self, path: str) -> int:
        tid = C.c_int32(-1)
        check(self.lib.ok_load_track_csv(self.h, path.encode(), C.byref(tid)))
        return tid.value

    def num_tracks(self) -> int:
        return self.lib.ok_num_tracks(self.h)

    def track_info(self, t: int) -> OkTrackInfo:
        info = OkTrackInfo()
        check(self.lib.ok_track_info(self.h, t, C.byref(info)))
        return info

    def track_array(self, t: int, name: str) -> np.ndarray:
        which = _capi.TRACK_ARRAYS[name]
        n = check(self.lib.ok_track_copy(self.h, t, which, None, 0))
        out = np.empty(n, dtype=np.float32)
        check(self.lib.ok_track_copy(self.h, t, which, _vp(out), n))
        if name in ("li", "lo", "ri", "ro"):
            return out.reshape(-1, 2)
        if name == "segments":
            return out.reshape(-1, 4)
        return out

    def beam_lookup(self, t: int, x: float, y: float, angle_rad: float):
        """OK_RAYCAST_BEAM's candidate list for a ray (host side): (segment indices nearest first, completeness
        distance), or None when the start cell is not covered by the table."""
        d = C.c_float(0.0)
        n = self.lib.ok_beam_lookup(self.h, t, x, y, angle_rad, None, 0, C.byref(d))
        if n == -100:  # OK_BEAM_NOT_COVERED
            return None
        check(n)
        items = np.empty(max(n, 1), dtype=np.uint16)
        check(self.lib.ok_beam_lookup(self.h, t, x, y, angle_rad, _vp(items), n, C.byref(d)))
        return items[:n], float(d.value)

    def beam_lookup_ex(self, t: int, x: float, y: float, angle_rad: float):
        """beam_lookup plus the first pass's view: (items, d_complete, d_inline, n_inline) or None"""
        d, d1, ni = C.c_float(0.0), C.c_float(0.0), C.c_int32(0)
        n = self.lib.ok_beam_lookup_ex(self.h, t, x, y, angle_rad, None, 0, C.byref(d), C.byref(d1), C.byref(ni))
        if n == -100:
            return None
        check(n)
        items = np.empty(max(n, 1), dtype=np.uint16)
        check(self.lib.ok_beam_lookup_ex(self.h, t, x, y, angle_rad, _vp(items), n, C.byref(d), C.byref(d1), C.byref(ni)))
        return items[:n], float(d.value), float(d1.value), int(ni.value)

    def beam_table_bytes(self, t: int) -> int:
        return check(self.lib.ok_beam_table_bytes(self.h, t))

    # ---- agents -------------------------------------------------------------------------
    def alloc_agents(self, n: int, ray_deg, track_id=None):
        ray_deg = np.ascontiguousarray(ray_deg, dtype=np.float32)
        tid = None if track_id is None else np.ascontiguousarray(track_id, dtype=np.int32)
        if tid is not None and len(tid) != n:
            raise ValueError("track_id must have one entry per agent")
        check(self.lib.ok_alloc_agents(self.h, n, len(ray_deg), _vp(ray_deg), _vp(tid)))
        self.n, self.rays = n, len(ray_deg)

    def reset(self, agent_idx, pt_idx, lane_alpha=None, heading_off=None, stream=None):
        """Host-array reset (Environment::resetAgent with explicit draws)."""
        ai = None if agent_idx is None else np.ascontiguousarray(agent_idx, dtype=np.int64)
        pt = np.ascontiguousarray(pt_idx, dtype=np.int32)
        la = None if lane_alpha is None else np.ascontiguousarray(lane_alpha, dtype=np.float32)
        ho = None if heading_off is None else np.ascontiguousarray(heading_off, dtype=np.float32)
        check(self.lib.ok_reset_agents_host(self.h, _vp(ai), _vp(pt), _vp(la), _vp(ho), len(pt), stream))

    def reset_device(self, d_agent_idx, d_pt_idx, d_lane_alpha, d_heading_off, n, stream=None):
        check(self.lib.ok_reset_agents(self.h, d_agent_idx, d_pt_idx, d_lane_alpha, d_heading_off, n, stream))

    # ---- reset draws (OkResetDraws: include/openkitchen_b200.h states the definition) -----
    def set_reset_draws(self, seed: int, point: bool = True, lane: bool = False, heading: bool = False):
        """Turn the reset draws on: with auto_reset the auto-reset of a crashed agent becomes a drawn reset, and
        reset_drawn / reset_drawn_device draw.  point / lane / heading: Environment::resetAgent's random centre-line point,
        lane lerp and +-(45..90) degree heading offset.  All three False turns the draws off."""
        flags = (_capi.RESET_DRAW_POINT if point else 0) | (_capi.RESET_DRAW_LANE if lane else 0) | (
            _capi.RESET_DRAW_HEADING if heading else 0)
        self.set_reset_draw_flags(seed, flags)

    def set_reset_draw_flags(self, seed: int, flags: int):
        """the same with the OK_RESET_DRAW_* bits (0 = off)"""
        flags = int(flags)
        if flags & ~(_capi.RESET_DRAW_POINT | _capi.RESET_DRAW_LANE | _capi.RESET_DRAW_HEADING):
            raise ValueError(f"unknown reset-draw flag bits in {flags:#x}")
        d = _capi.OkResetDraws(seed=int(seed) & 0xFFFFFFFF, flags=flags)
        check(self.lib.ok_set_reset_draws(self.h, C.byref(d)))

    def reset_draws(self) -> dict:
        """{"seed", "point", "lane", "heading"} as set; every flag False = off"""
        d = _capi.OkResetDraws()
        check(self.lib.ok_get_reset_draws(self.h, C.byref(d)))
        return {"seed": int(d.seed), "point": bool(d.flags & _capi.RESET_DRAW_POINT),
                "lane": bool(d.flags & _capi.RESET_DRAW_LANE), "heading": bool(d.flags & _capi.RESET_DRAW_HEADING)}

    def _drawn_args(self, agent_idx, mask):
        if agent_idx is not None and mask is not None:
            raise ValueError("pass agent indices or a mask, not both")
        if agent_idx is not None:
            ai = np.ascontiguousarray(agent_idx, dtype=np.int64).reshape(-1)
            return ai, None, len(ai)
        if mask is not None:
            m = np.ascontiguousarray(mask).reshape(-1)
            if len(m) != self.n:
                raise ValueError(f"the mask must have one entry per agent ({self.n}), got {len(m)}")
            return None, m.astype(np.uint8), self.n
        return None, None, self.n

    def reset_drawn(self, agent_idx=None, mask=None, stream=None):
        """Drawn reset (host arrays) of the agents agent_idx, of those where mask is set (one entry per agent), or of all
        agents.  Synchronises `stream`."""
        ai, m, n = self._drawn_args(agent_idx, mask)
        check(self.lib.ok_reset_agents_drawn_host(self.h, _vp(ai), _vp(m), n, stream))

    def reset_drawn_device(self, d_agent_idx=None, d_mask=None, n=None, stream=None):
        """device-pointer form of reset_drawn (asynchronous on `stream`): d_agent_idx i64[n], or d_mask u8[agents], or
        neither (all agents); n defaults to the agent count"""
        if d_agent_idx and d_mask:
            raise ValueError("pass agent indices or a mask, not both")
        if n is None:
            if d_agent_idx:
                raise ValueError("n is required with agent indices")
            n = self.n
        elif not d_agent_idx and n != self.n:
            raise ValueError(f"with a mask or for all agents, n must be the agent count ({self.n})")
        check(self.lib.ok_reset_agents_drawn(self.h, d_agent_idx, d_mask, n, stream))

    def reset_draw_counts_info(self):
        """(device pointer, shape, dtype) of the reset-draw counters k, u32[agents]"""
        ptr = C.c_void_p()
        check(self.lib.ok_reset_draw_counts(self.h, C.byref(ptr)))
        return ptr.value, (self.n,), np.uint32

    # ---- lap accounting (OkLaps: include/openkitchen_b200.h states the definition) -------
    def set_laps(self, target: int = 0, enabled: bool = True, stream=None):
        """Lap accounting on (or off with enabled=False): every moving tick adds the agent's signed centre-line progress,
        counts laps of P points from where its episode started and their lengths in ticks, and with target > 0 sets the
        agent's completed flag (and so done) at `target` laps; with auto_reset a completed agent is reset.  target 0 =
        never complete.  Switching it on restarts every agent's lap state (asynchronous on `stream`)."""
        target = int(target)
        if target < 0:
            raise ValueError("the lap target must be >= 0")
        check(self.lib.ok_set_laps(self.h, C.byref(_capi.OkLaps(enabled=1 if enabled else 0, target=target)), stream))

    def laps(self) -> dict:
        """{"enabled", "target"} as set"""
        l = _capi.OkLaps()
        check(self.lib.ok_get_laps(self.h, C.byref(l)))
        return {"enabled": bool(l.enabled), "target": int(l.target)}

    def lap_buffers_info(self) -> dict:
        """{field: (device pointer, shape, dtype)} of the seven lap arrays (OkLapBuffers), [agents] each"""
        b = _capi.OkLapBuffers()
        check(self.lib.ok_lap_buffers(self.h, C.byref(b)))
        return {f: (getattr(b, f), (self.n,), np.dtype(dt).type) for f, dt in _capi.LAP_ARRAYS.items()}

    # ---- races (OkRaces: include/openkitchen_b200.h states the definition) ---------------
    def set_races(self, group: int, radius: float = 0.0, sense: bool = True, contact: bool = True):
        """Races on: agents a // group race each other.  A car is a disc of `radius` px around its position; with `sense`
        the lidar sees the opponents on its track, with `contact` overlapping cars crash.  A pass after every tick that
        casts rays does both; a car it crashes has crashed, done and contact set.  group 0 turns races off."""
        group = int(group)
        flags = (_capi.RACE_SENSE if sense else 0) | (_capi.RACE_CONTACT if contact else 0)
        if group and not (2 <= group <= 1024):
            raise ValueError("the race group must be 0 (off) or in 2..1024")
        if group and not (np.isfinite(radius) and radius > 0):
            raise ValueError("the car radius must be finite and > 0")
        if group and not flags:
            raise ValueError("a race needs sense, contact or both")
        check(self.lib.ok_set_races(self.h, C.byref(_capi.OkRaces(group=group, flags=flags, radius=float(radius)))))

    def races(self) -> dict:
        """{"group", "radius", "sense", "contact"} as set; group 0 = off"""
        r = _capi.OkRaces()
        check(self.lib.ok_get_races(self.h, C.byref(r)))
        return {"group": int(r.group), "radius": float(r.radius), "sense": bool(r.flags & _capi.RACE_SENSE),
                "contact": bool(r.flags & _capi.RACE_CONTACT)}

    def race_buffers_info(self) -> dict:
        """{"hit_car": (device pointer, (agents, rays), int32), "contact": (pointer, (agents,), uint8)} (OkRaceBuffers);
        they exist once races have been switched on for this population"""
        b = _capi.OkRaceBuffers()
        check(self.lib.ok_race_buffers(self.h, C.byref(b)))
        return {"hit_car": (b.hit_car, (self.n, self.rays), np.int32), "contact": (b.contact, (self.n,), np.uint8)}

    # ---- the tick -----------------------------------------------------------------------
    def cast_rays(self, stream=None):
        check(self.lib.ok_cast_rays(self.h, stream))

    def launch_step(self, d_thr=None, d_steer=None, stream=None):
        check(self.lib.ok_launch_step(self.h, d_thr, d_steer, stream))

    def launch_steps_random(self, first_step: int, k: int, seed: int = 0x0C17C4E2, stream=None):
        check(self.lib.ok_launch_steps_random(self.h, first_step, k, seed, stream))

    def fill_random_actions(self, step: int, seed: int = 0x0C17C4E2, stream=None):
        check(self.lib.ok_fill_random_actions(self.h, step, seed, stream))

    def genetic_policy(self, d_w1, d_w2, hidden: int, stream=None):
        """per-agent shallow MLP -> ACT_* buffers (device weight pointers)"""
        check(self.lib.ok_genetic_policy(self.h, d_w1, d_w2, hidden, stream))

    def cmaes_controller(self, d_params, n_params: int, hidden: int = 16, throttle: float = 100.0, steer_scale: float = 5.0,
                         stream=None):
        """per-candidate Controller MLP -> ACT_* buffers (device pointer to f32[N, n_params])"""
        check(self.lib.ok_cmaes_controller(self.h, d_params, n_params, hidden, throttle, steer_scale, stream))

    def ppo_actor(self, io, step: int = 0, seed: int = 0x0C17C4E2, stream=None):
        """obs -> actor MLP -> softmax -> sample -> action buffers, one kernel (io: _capi.OkActorIO of device pointers)"""
        check(self.lib.ok_ppo_actor(self.h, C.byref(io), step, seed, stream))

    def ppo_actor_step(self, io, step: int = 0, seed: int = 0x0C17C4E2, stream=None):
        """ppo_actor + the tick that consumes its actions as ONE launch (ok_ppo_actor_step)"""
        check(self.lib.ok_ppo_actor_step(self.h, C.byref(io), step, seed, stream))

    def discounted_returns(self, d_rewards, d_done, d_out, steps: int, n: int, gamma: float = 0.99, stream=None):
        check(self.lib.ok_discounted_returns(self.h, d_rewards, d_done, d_out, steps, n, gamma, stream))

    def step_host(self, thr=None, steer=None, obs=None, reward=None, done=None, stream=None):
        """End-to-end tick with HOST buffers (H2D actions, kernel, D2H results, sync).  An `obs` array of dtype uint16
        selects the opt-in, LOSSY 16-bit fixed-point observations (ok_step_host_q16: rn(clamp(obs, 0, 1) * 65535))."""
        if obs is not None and getattr(obs, "dtype", None) == np.uint16:
            check(self.lib.ok_step_host_q16(self.h, _vp(thr), _vp(steer), _vp(obs), _vp(reward), _vp(done), stream))
        else:
            check(self.lib.ok_step_host(self.h, _vp(thr), _vp(steer), _vp(obs), _vp(reward), _vp(done), stream))

    def track_query(self, x, y, track_id=None, stream=None):
        """RaceTrack::findNearestTrackIndexBruteForce / getDistanceToLaneCenter / getNearestDistanceToTrackBoundary
        (RaceTrack.cpp:16-72) for host arrays of points -> (nearest_idx i32[n], dist_lane_center f32[n],
        dist_boundary f32[n]), computed on the device."""
        x = np.ascontiguousarray(x, dtype=np.float32)
        y = np.ascontiguousarray(y, dtype=np.float32)
        if x.shape != y.shape or x.ndim != 1:
            raise ValueError("x and y must be 1-d arrays of one length")
        t = None if track_id is None else np.ascontiguousarray(track_id, dtype=np.int32)
        idx = np.empty(len(x), dtype=np.int32)
        lane = np.empty(len(x), dtype=np.float32)
        bound = np.empty(len(x), dtype=np.float32)
        check(self.lib.ok_track_query_host(self.h, _vp(x), _vp(y), _vp(t), len(x), _vp(idx), _vp(lane), _vp(bound), stream))
        return idx, lane, bound

    def track_query_device(self, d_x, d_y, d_track_id, n, d_idx=None, d_lane=None, d_bound=None, stream=None):
        """device-pointer form (asynchronous on `stream`)"""
        check(self.lib.ok_track_query(self.h, d_x, d_y, d_track_id, n, d_idx, d_lane, d_bound, stream))

    def lidar_query(self, x, y, rot, track_id=None, ray_deg=None, stream=None) -> dict:
        """Lidar scans at arbitrary poses (host arrays), with no agent state read or written: what ok_cast_rays would give
        agents at these poses with their crash flags clear.  ray_deg None = the fan of alloc_agents.  Returns a dict keyed
        by the BatchEnv names (see LIDAR_OUTPUTS); synchronises `stream`."""
        x, y, rot = _pose_arrays(x, y, rot, track_id)
        t = None if track_id is None else np.ascontiguousarray(track_id, dtype=np.int32)
        fan = None if ray_deg is None else np.ascontiguousarray(ray_deg, dtype=np.float32).reshape(-1)
        n, rays = len(x), (self.rays if fan is None else len(fan))
        out = {name: np.empty(shape(n, rays), dtype=dt) for name, (_, dt, shape) in LIDAR_OUTPUTS.items()}
        q = _capi.OkLidarQuery(x=_vp(x), y=_vp(y), rot=_vp(rot), track_id=_vp(t), n=n, ray_deg=_vp(fan), rays=rays)
        for name, (field, _, _) in LIDAR_OUTPUTS.items():
            setattr(q, field, _vp(out[name]))
        check(self.lib.ok_lidar_query_host(self.h, C.byref(q), stream))
        return out

    def lidar_query_device(self, d_x, d_y, d_rot, n: int, d_track_id=None, d_ray_deg=None, rays=None, stream=None, **d_out):
        """device-pointer form of lidar_query (asynchronous on `stream`): d_out maps the C field names (hit_abs, hit_rel,
        obs, hit_t, hit_seg, min_dist2, crashed) to device pointers; absent outputs are not computed.  rays None = the
        env's ray count."""
        fields = {f for f, _, _ in LIDAR_OUTPUTS.values()}
        unknown = set(d_out) - fields
        if unknown:
            raise ValueError(f"unknown lidar outputs {sorted(unknown)}; expected some of {sorted(fields)}")
        q = _capi.OkLidarQuery(x=d_x, y=d_y, rot=d_rot, track_id=d_track_id, n=n, ray_deg=d_ray_deg,
                               rays=self.rays if rays is None else rays, **d_out)
        check(self.lib.ok_lidar_query(self.h, C.byref(q), stream))

    def bev_query(self, x, y, rot, height: int, width: int, scale: float, ahead: float = 0.0, track_id=None,
                  stream=None) -> np.ndarray:
        """Bird's-eye-view rasters at arbitrary poses (host arrays), with no agent state read or written: u8[n, height,
        width] of BEV_OFF / BEV_WALL / BEV_LANE, row 0 ahead, column 0 on the left; `scale` track px per image pixel,
        `ahead` px forward (ok_bev_query_host; the header states the exact definition).  Synchronises `stream`."""
        x, y, rot = _pose_arrays(x, y, rot, track_id)
        height, width, scale, ahead = _bev_shape(height, width, scale, ahead)
        if self.num_tracks() == 0:
            raise ValueError("no track has been added")
        t = None if track_id is None else np.ascontiguousarray(track_id, dtype=np.int32)
        out = np.empty((len(x), height, width), dtype=np.uint8)
        q = _capi.OkBevQuery(x=_vp(x), y=_vp(y), rot=_vp(rot), track_id=_vp(t), n=len(x), height=height, width=width,
                             scale=scale, ahead=ahead, out=_vp(out))
        check(self.lib.ok_bev_query_host(self.h, C.byref(q), stream))
        return out

    def bev_query_device(self, d_x, d_y, d_rot, n: int, height: int, width: int, scale: float, d_out, ahead: float = 0.0,
                         d_track_id=None, stream=None):
        """device-pointer form of bev_query (asynchronous on `stream`): d_out is u8[n, height, width]"""
        height, width, scale, ahead = _bev_shape(height, width, scale, ahead)
        if n < 0:
            raise ValueError("n < 0")
        if n > 0 and not (d_x and d_y and d_rot and d_out):
            raise ValueError("pose and output pointers must not be NULL")
        if self.num_tracks() == 0:
            raise ValueError("no track has been added")
        q = _capi.OkBevQuery(x=d_x, y=d_y, rot=d_rot, track_id=d_track_id, n=n, height=height, width=width, scale=scale,
                             ahead=ahead, out=d_out)
        check(self.lib.ok_bev_query(self.h, C.byref(q), stream))

    def sync(self, stream=None):
        check(self.lib.ok_sync(self.h, stream))

    # ---- buffers ------------------------------------------------------------------------
    def buffer_info(self, name: str):
        """(device pointer, shape tuple, numpy dtype) of an agent buffer."""
        ptr, shape, dt = C.c_void_p(), (C.c_int64 * 3)(), C.c_int32()
        check(self.lib.ok_get_buffer(self.h, BUF[name], C.byref(ptr), shape, C.byref(dt)))
        shp = tuple(int(s) for s in shape if s > 0)
        return ptr.value, shp, _NP_DTYPES[dt.value]

    def read(self, name: str, stream=None) -> np.ndarray:
        _, shp, dt = self.buffer_info(name)
        out = np.empty(shp, dtype=dt)
        check(self.lib.ok_read_buffer(self.h, BUF[name], _vp(out), out.nbytes, stream))
        return out

    def write(self, name: str, arr, stream=None):
        _, shp, dt = self.buffer_info(name)
        a = np.ascontiguousarray(arr, dtype=dt)
        if a.shape != shp:
            raise ValueError(f"{name}: expected shape {shp}, got {a.shape}")
        check(self.lib.ok_write_buffer(self.h, BUF[name], _vp(a), a.nbytes, stream))

    def eval_sincosf(self, x):
        """the device sincosf on host floats -> (sin, cos); for tests of the arithmetic model"""
        x = np.ascontiguousarray(x, dtype=np.float32)
        s, c = np.empty_like(x), np.empty_like(x)
        check(self.lib.ok_eval_sincosf(self.h, _vp(x), _vp(s), _vp(c), x.size))
        return s, c

    def debug_stats(self, enable: bool = True):
        """(rays cast, rays queued for the second pass, rays sent to the grid walk) since the previous call"""
        out = (C.c_uint64 * 4)()
        check(self.lib.ok_debug_stats(self.h, out, 1 if enable else 0))
        return int(out[0]), int(out[1]), int(out[2])

    def debug_violations(self):
        """(out-of-range indices counted by an OK_CHECKED build, whether this library was built with the checks)"""
        n, on = C.c_uint64(0), C.c_int32(0)
        check(self.lib.ok_debug_violations(self.h, C.byref(n), C.byref(on)))
        return int(n.value), bool(on.value)

    def debug_trace(self, tiles_per_cta: int = 0):
        """timeline of the last beam-kernel launch as u64[grid, tiles, 6] (None if tracing was off); then re-arms the
        trace for `tiles_per_cta` tiles per CTA (0 = off)"""
        grid = self.launch_stats().grid_blocks
        cap = grid * 64 * 6
        buf = np.zeros(cap, dtype=np.uint64)
        got = check(self.lib.ok_debug_trace(self.h, _vp(buf), cap, tiles_per_cta))
        return buf[:got].reshape(grid, -1, 6) if got else None

    def balance_schedule(self, stream: int = 0):
        """re-cuts the beam kernel's tiles from the tile times of the last launch (ok_balance_schedule); returns
        (slowest tile / mean tile before, predicted after).  The library also does this on its own early in a run."""
        out = (C.c_float * 2)()
        check(self.lib.ok_balance_schedule(self.h, C.c_void_p(stream), out))
        return float(out[0]), float(out[1])

    def debug_tiles(self) -> np.ndarray:
        """the beam kernel's tiling as i64[tiles, 3] = {track, count, first agent} (ok_debug_trace's tile ids index it)"""
        n = check(self.lib.ok_debug_tiles(self.h, None, 0))
        buf = np.zeros((max(n, 1), 3), dtype=np.int64)
        check(self.lib.ok_debug_tiles(self.h, _vp(buf), n))
        return buf[:n]

    def population_counters(self, stream=None) -> dict:
        """agents / alive / crashed / timed_out / done right now, counted on the device (ok_population_counters)"""
        c = OkPopulationCounters()
        check(self.lib.ok_population_counters(self.h, C.byref(c), stream))
        return {k: int(getattr(c, k)) for k, _ in c._fields_}

    def launch_stats(self) -> OkLaunchStats:
        s = OkLaunchStats()
        check(self.lib.ok_launch_stats(self.h, C.byref(s)))
        return s


def quantize_obs_q16(obs) -> np.ndarray:
    """the fixed point ok_step_host_q16 delivers, from float observations: rn(clamp(obs, 0, 1) * 65535) in binary32 -- the
    host-side statement of the kernel's obs_q16 (tests compare the two)"""
    o = np.clip(np.asarray(obs, dtype=np.float32), np.float32(0), np.float32(1))
    return np.rint(o * np.float32(65535.0)).astype(np.uint16)


def dequantize_obs_q16(q) -> np.ndarray:
    """float32 observations (norm / sensor range, in [0, 1]) from ok_step_host_q16's uint16; |error| <= 0.5 / 65535 of the range"""
    return (np.asarray(q, dtype=np.uint16).astype(np.float32) / np.float32(65535.0)).astype(np.float32)


def pcie_probe(device: int, nbytes: int, iters: int = 50, mode: str = "d2h") -> float:
    """GB/s of `iters` transfers of `nbytes` between pinned host memory and `device` (measurement only):
    mode "d2h" = DMA copies, "store" = kernel stores through the host mapping, "h2d" = DMA copies the other way"""
    g = C.c_double(0.0)
    check(_capi.load().ok_pcie_probe(device, nbytes, iters, {"d2h": 0, "store": 1, "h2d": 2}[mode], C.byref(g)))
    return g.value


def pinned_array(shape, dtype) -> np.ndarray:
    """numpy array over cudaMallocHost memory (for the end-to-end path); freed when collected."""
    lib = _capi.load()
    nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
    p = C.c_void_p()
    check(lib.ok_host_alloc(C.byref(p), max(nbytes, 1)))
    buf = (C.c_uint8 * max(nbytes, 1)).from_address(p.value)
    arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    class _Owner:
        def __init__(self, ptr):
            self.ptr = ptr

        def __del__(self):
            try:
                lib.ok_host_free(self.ptr)
            except Exception:
                pass

    _OWNERS[id(buf)] = _Owner(p)  # keep alive as long as the module (simple and safe for benches)
    return arr


_OWNERS = {}

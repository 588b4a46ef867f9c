"""``BatchEnv``: the batch API the Python RL / evolution trainers use (SURVEY.md section 8b, "Python" row).

All state lives on the GPU; every attribute is a ZERO-COPY ``torch`` view (via DLPack) of the buffers the
kernels read and write, on torch's current CUDA stream.  A policy writes ``env.actions`` (or passes action
tensors to ``step``), calls ``env.step()`` and reads ``env.obs`` / ``env.reward`` / ``env.done`` -- nothing
crosses PCIe.  Replaces the reference's per-agent host loop of ``torch::tensor(getCurrentState())`` +
``.item()`` (RLRacers/PPO/PPOAgent.hpp:68-102) and ``Pybind/bindings.cpp``'s single-agent ``BoundEnv``.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _capi
from .dlpack import DeviceBuffer
from .env import LIDAR_OUTPUTS, Env, _bev_shape, ray_fan, track_names

_TORCH_DTYPES = {np.float32: torch.float32, np.int32: torch.int32, np.uint8: torch.uint8}


class BatchEnv:
    def __init__(self, tracks, n_agents: int, rays=32, device=0, track_id=None, **cfg):
        """tracks: names from the packed racetrack-database set, CSV paths, or (x, y, w_right, w_left)
        column tuples.  rays: a count (evenly spaced -70..70 deg fan) or explicit angles in degrees."""
        if isinstance(device, torch.device):
            device = device.index or 0
        self.device = torch.device("cuda", int(device))
        self.env = Env(device=int(device), **cfg)
        known = set(track_names())
        for t in ([tracks] if isinstance(tracks, str) else tracks):
            if isinstance(t, str):
                self.env.add_named_track(t) if t in known else self.env.load_track_csv(t)
            else:
                self.env.add_track(t)
        nt = self.env.num_tracks()
        fan = ray_fan(rays) if np.isscalar(rays) else np.asarray(rays, dtype=np.float32)
        if track_id is None:
            track_id = (np.arange(n_agents, dtype=np.int64) * nt // n_agents).astype(np.int32)
        self.env.alloc_agents(n_agents, fan, track_id)
        self.n_agents, self.n_rays = n_agents, len(fan)
        self.track_id = torch.as_tensor(np.asarray(track_id, dtype=np.int32))
        self.points_per_track = [self.env.track_info(t).n_points for t in range(nt)]
        self._views = {}
        for name in _capi.BUFFERS:
            self._views[name] = torch.from_dlpack(DeviceBuffer(self.env, name))
        v = self._views
        # the reference's names for things
        self.obs = v["obs"]                  # f32[N,R]  sensor_hits_[i].norm() / kSensorRange
        self.hits = v["hit_rel"]             # f32[N,R,2] Agent::sensor_hits_
        self.hit_points = v["hit_abs"]       # f32[N,R,2] Ray_::hit_x / hit_y
        self.hit_seg = v["hit_seg"]          # i32[N,R]
        self.hit_t = v["hit_t"]              # f32[N,R]
        self.reward = v["reward"]
        self.fitness = v["fitness"]
        self.done = v["done"]
        self.crashed = v["crashed"]
        self.timed_out = v["timed_out"]
        self.nearest_idx = v["nearest_idx"]
        self.pos_x, self.pos_y, self.rot, self.speed = v["pos_x"], v["pos_y"], v["rot"], v["speed"]
        self.act_throttle, self.act_steer = v["act_throttle"], v["act_steer"]
        # u32[N]: the reset-draw counters k (set_reset_draws); not an OkBuffer, so not in ok.BUFFERS / self[name]
        self.reset_draw_count = torch.from_dlpack(DeviceBuffer(self.env, "reset_draw_count", self.env.reset_draw_counts_info()))
        # [N] each: the lap-accounting state (set_laps; OkLaps in include/openkitchen_b200.h), also not OkBuffers
        lap = {f: torch.from_dlpack(DeviceBuffer(self.env, f, info)) for f, info in self.env.lap_buffers_info().items()}
        self.lap_idx = lap["lap_idx"]            # i32: centre-line index at which progress was last measured
        self.lap_progress = lap["progress"]      # i32: signed centre-line points since the episode started
        self.laps = lap["laps"]                  # i32: laps completed
        self.lap_ticks = lap["ticks"]            # u32: ticks moved since the episode started
        self.lap_start_ticks = lap["lap_start"]  # u32: lap_ticks when the current lap began
        self.last_lap_ticks = lap["last_lap"]    # u32: ticks of the last completed lap, 0 = none yet
        self.completed = lap["completed"]        # u8: Agent::completed_ (laps >= target)
        # the race pass's outputs (set_races; OkRaces in include/openkitchen_b200.h), not OkBuffers either: they exist once
        # races have been switched on, and are None until then
        self.hit_car = None  # i32[N,R]: the opponent a ray hit, -1 = none
        self.contact = None  # u8[N]: crashed by the last race pass
        self._step_count = 0

    # ---- views -----------------------------------------------------------------------------
    def __getitem__(self, name: str) -> torch.Tensor:
        return self._views[name]

    @property
    def pose(self) -> torch.Tensor:
        """f32[N,4] = (x, y, rot_deg, speed), a fresh stack (the state itself is structure-of-arrays)"""
        return torch.stack([self.pos_x, self.pos_y, self.rot, self.speed], dim=1)

    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    # ---- the tick --------------------------------------------------------------------------
    def step(self, throttle: torch.Tensor | None = None, steer: torch.Tensor | None = None, k: int = 1):
        """One tick (k ticks with the same action).  throttle/steer: f32[N] CUDA tensors; None = use
        ``act_throttle`` / ``act_steer`` as they are (what ``Agent::updateAction`` left there)."""
        if (throttle is None) != (steer is None):
            raise ValueError("pass both action tensors or neither")
        dt = ds = None
        if throttle is not None:
            throttle = throttle.to(self.device, torch.float32).contiguous()
            steer = steer.to(self.device, torch.float32).contiguous()
            if throttle.numel() != self.n_agents or steer.numel() != self.n_agents:
                raise ValueError("one action per agent")
            dt, ds = throttle.data_ptr(), steer.data_ptr()
        for _ in range(k):
            self.env.launch_step(dt, ds, self._stream())
        self._step_count += k
        return self.obs, self.reward, self.done

    def step_random(self, k: int = 1, seed: int = 0x0C17C4E2):
        """k ticks driven by the counter-based Philox action stream generated inside the kernel"""
        self.env.launch_steps_random(self._step_count, k, seed, self._stream())
        self._step_count += k
        return self.obs, self.reward, self.done

    def cast_rays(self):
        self.env.cast_rays(self._stream())
        return self.obs

    def lidar(self, x, y, rot, track_id=None, rays=None, outputs=None) -> dict:
        """Lidar scans at arbitrary poses, with no agent state read or written (ok_lidar_query): what ``cast_rays`` would
        give agents at these poses with their crash flags clear.  x, y, rot: f32[n] (rot in degrees); track_id: i32[n] or
        None (track 0).  rays: None (this env's fan), a count or angles, as in the constructor.  outputs: names to compute
        (default all of obs, hits, hit_points, hit_seg, hit_t, min_dist2, crashed).  Returns fresh tensors keyed by those
        names, computed on torch's current stream with no host synchronisation."""
        names = list(LIDAR_OUTPUTS) if outputs is None else list(outputs)
        unknown = [nm for nm in names if nm not in LIDAR_OUTPUTS]
        if unknown:
            raise ValueError(f"unknown lidar outputs {unknown}; expected some of {list(LIDAR_OUTPUTS)}")
        n = int(torch.as_tensor(x).numel())
        if any(torch.as_tensor(a).dim() != 1 for a in (x, y, rot)) or any(int(torch.as_tensor(a).numel()) != n for a in (y, rot)):
            raise ValueError("x, y and rot must be 1-d tensors of one length")
        if track_id is not None and int(torch.as_tensor(track_id).numel()) != n:
            raise ValueError("track_id must have one entry per pose")
        x, y, rot = (torch.as_tensor(a).to(self.device, torch.float32).contiguous() for a in (x, y, rot))
        tid = None if track_id is None else torch.as_tensor(track_id).to(self.device, torch.int32).contiguous()
        fan = None if rays is None else self._fan(rays)
        r = self.n_rays if fan is None else int(fan.numel())
        out = {nm: torch.empty(LIDAR_OUTPUTS[nm][2](n, r), device=self.device, dtype=_TORCH_DTYPES[LIDAR_OUTPUTS[nm][1]])
               for nm in names}
        self.env.lidar_query_device(x.data_ptr(), y.data_ptr(), rot.data_ptr(), n, None if tid is None else tid.data_ptr(),
                                    None if fan is None else fan.data_ptr(), r, self._stream(),
                                    **{LIDAR_OUTPUTS[nm][0]: t.data_ptr() for nm, t in out.items()})
        return out

    def bev(self, height: int = 64, width: int = 64, scale: float = 1.0, ahead: float = 0.0, x=None, y=None, rot=None,
            track_id=None) -> torch.Tensor:
        """Bird's-eye-view rasters (ok_bev_query): u8[n, height, width] of ok.BEV_OFF / BEV_WALL / BEV_LANE around each
        pose, row 0 ahead, column 0 on the left, `scale` track px per image pixel, the image shifted `ahead` px forward.
        The poses default to the population's own pos_x / pos_y / rot / track_id; x, y, rot: f32[n] (rot in degrees),
        track_id: i32[n] or None (track 0 for explicit poses).  Returns a fresh tensor, computed on torch's current stream
        with no host synchronisation."""
        height, width, scale, ahead = _bev_shape(height, width, scale, ahead)
        if x is None and y is None and rot is None:
            x, y, rot = self.pos_x, self.pos_y, self.rot
            if track_id is None:
                track_id = self._views["track_id"]
        elif x is None or y is None or rot is None:
            raise ValueError("pass all of x, y and rot, or none of them")
        n = int(torch.as_tensor(x).numel())
        if any(torch.as_tensor(a).dim() != 1 for a in (x, y, rot)) or any(int(torch.as_tensor(a).numel()) != n for a in (y, rot)):
            raise ValueError("x, y and rot must be 1-d tensors of one length")
        if track_id is not None and int(torch.as_tensor(track_id).numel()) != n:
            raise ValueError("track_id must have one entry per pose")
        x, y, rot = (torch.as_tensor(a).to(self.device, torch.float32).contiguous() for a in (x, y, rot))
        tid = None if track_id is None else torch.as_tensor(track_id).to(self.device, torch.int32).contiguous()
        out = torch.empty((n, height, width), device=self.device, dtype=torch.uint8)
        self.env.bev_query_device(x.data_ptr(), y.data_ptr(), rot.data_ptr(), n, height, width, scale, out.data_ptr(), ahead,
                                  None if tid is None else tid.data_ptr(), self._stream())
        return out

    def _fan(self, rays) -> torch.Tensor:
        """a ray fan as a device tensor, kept per distinct fan: the upload happens once, later queries do not wait for it"""
        a = ray_fan(rays) if np.isscalar(rays) else np.ascontiguousarray(torch.as_tensor(rays).cpu().numpy(), dtype=np.float32)
        key = a.tobytes()
        fans = self.__dict__.setdefault("_fans", {})
        if key not in fans:
            fans[key] = torch.from_numpy(a.copy()).to(self.device)
        return fans[key]

    # ---- resets ----------------------------------------------------------------------------
    def reset(self, agents=None, pt_idx=None, lane_alpha=None, heading_off=None):
        """Environment::resetAgent with explicit draws.  agents: None (all), a bool mask or an index tensor.
        pt_idx None = RaceTrack::kStartingIdx (3).  All arguments may be CUDA tensors (no host sync)."""
        if agents is None:
            idx = torch.arange(self.n_agents, device=self.device, dtype=torch.int64)
        else:
            agents = torch.as_tensor(agents, device=self.device)
            idx = torch.nonzero(agents, as_tuple=False).flatten() if agents.dtype == torch.bool else agents.to(torch.int64)
        n = int(idx.numel())
        if n == 0:
            return
        if pt_idx is None:
            pt = torch.full((n,), 3, device=self.device, dtype=torch.int32)
        else:
            pt = torch.as_tensor(pt_idx, device=self.device).to(torch.int32).contiguous()
        la = None if lane_alpha is None else torch.as_tensor(lane_alpha, device=self.device).to(torch.float32).contiguous()
        ho = None if heading_off is None else torch.as_tensor(heading_off, device=self.device).to(torch.float32).contiguous()
        idx = idx.contiguous()
        self.env.reset_device(idx.data_ptr(), pt.data_ptr(), None if la is None else la.data_ptr(),
                              None if ho is None else ho.data_ptr(), n, self._stream())
        self._keep = (idx, pt, la, ho)  # alive until the kernel has run

    def reset_random(self, agents=None, generator: torch.Generator | None = None, randomize_lane=False,
                     randomize_heading=False):
        """Environment::resetAgent(agent, true, lane, heading) (Environment.cpp:79-122) with torch's RNG standing
        in for raylib's GetRandomValue: idx ~ U{0..P-1}, alpha ~ U{10..90}/100, offset ~ +-(45 + U{0..45})."""
        if agents is None:
            idx = torch.arange(self.n_agents, device=self.device)
        else:
            agents = torch.as_tensor(agents, device=self.device)
            idx = torch.nonzero(agents, as_tuple=False).flatten() if agents.dtype == torch.bool else agents.to(torch.int64)
        n = int(idx.numel())
        if n == 0:
            return
        pts = torch.as_tensor(self.points_per_track, device=self.device)[self.track_id.to(self.device)[idx].long()]
        u = torch.rand(n, device=self.device, generator=generator)
        pt = torch.minimum((u * pts).to(torch.int32), (pts - 1).to(torch.int32))
        la = ho = None
        if randomize_lane:
            la = torch.randint(10, 91, (n,), device=self.device, generator=generator).float() / 100.0
        if randomize_heading:
            mag = 45.0 + torch.randint(0, 46, (n,), device=self.device, generator=generator).float()
            sign = torch.where(torch.arange(n, device=self.device) % 2 == 0, -1.0, 1.0)
            ho = mag * sign
        self.reset(idx, pt, la, ho)

    def set_reset_draws(self, seed: int, point: bool = True, lane: bool = False, heading: bool = False):
        """Reset draws (include/openkitchen_b200.h, OkResetDraws): Environment::resetAgent's random centre-line point, lane
        lerp and heading offset from a counter-based stream keyed by (seed, agent id, reset_draw_count[agent]).  With
        auto_reset the tick's own reset of crashed agents draws, inside the step kernel, so a captured rollout starts its
        episodes where the reference's apps would; reset_drawn draws too.  All three False turns the draws off."""
        self.env.set_reset_draws(seed, point, lane, heading)

    def reset_draws(self) -> dict:
        return self.env.reset_draws()

    def set_laps(self, target: int = 0, enabled: bool = True):
        """Lap accounting (include/openkitchen_b200.h, OkLaps): every moving tick adds the agent's signed centre-line
        progress to lap_progress, counts laps of P centre-line points from where its episode started (laps) and their
        lengths in ticks (last_lap_ticks); with target > 0 an agent's completed flag, and so done, is set at `target` laps,
        and auto_reset resets it like a crashed agent.  All inside the step kernel.  Switching it on restarts every agent's
        lap state on torch's current stream; enabled=False turns it off (the tick then leaves the arrays alone)."""
        self.env.set_laps(target, enabled, self._stream())

    def lap_settings(self) -> dict:
        """{"enabled", "target"} as set"""
        return self.env.laps()

    def set_races(self, group: int, radius: float = 0.0, sense: bool = True, contact: bool = True):
        """Races (include/openkitchen_b200.h, OkRaces): agents a // group race each other, as discs of `radius` px on the
        same track.  After every tick a pass on torch's current stream lets the lidar see the opponents (sense: a nearer car
        replaces the track hit, hit_car names it, and min_dist2's crash rule applies to it) and crashes overlapping cars
        (contact).  A car the pass crashes has crashed, done and contact set; reward is the track-only reward, so a penalty
        is one op: ``env.reward[env.contact.bool()] -= p``.  group 0 turns races off."""
        self.env.set_races(group, radius, sense, contact)
        if self.hit_car is None and int(group):
            bufs = self.env.race_buffers_info()
            self.hit_car = torch.from_dlpack(DeviceBuffer(self.env, "hit_car", bufs["hit_car"]))
            self.contact = torch.from_dlpack(DeviceBuffer(self.env, "contact", bufs["contact"]))

    def race_settings(self) -> dict:
        """{"group", "radius", "sense", "contact"} as set; group 0 = off"""
        return self.env.races()

    def reset_drawn(self, agents=None):
        """Drawn reset (ok_reset_agents_drawn) of agents: None (all), a bool / uint8 CUDA mask with one entry per agent (e.g.
        ``env.done``, passed as it is: no nonzero, no host synchronisation), or an index tensor.  Runs on torch's current
        stream; it can be captured into a CUDA graph."""
        if agents is None:
            self.env.reset_drawn_device(None, None, self.n_agents, self._stream())
            return
        agents = torch.as_tensor(agents, device=self.device)
        if agents.dtype in (torch.bool, torch.uint8):
            if agents.numel() != self.n_agents:
                raise ValueError(f"the mask must have one entry per agent ({self.n_agents}), got {agents.numel()}")
            mask = agents.contiguous()
            if mask.dtype == torch.bool:
                mask = mask.view(torch.uint8)  # same bytes: 0 / 1
            self.env.reset_drawn_device(None, mask.data_ptr(), self.n_agents, self._stream())
            self._keep_drawn = mask
            return
        idx = agents.to(torch.int64).contiguous().reshape(-1)
        if idx.numel() == 0:
            return
        self.env.reset_drawn_device(idx.data_ptr(), None, int(idx.numel()), self._stream())
        self._keep_drawn = idx  # alive until the kernel has run

    def close(self):
        """Drops this object's views and closes the env.  Tensors the caller still holds keep the device memory alive:
        the OkEnv is destroyed when the last of them is released (openkitchen_b200.dlpack)."""
        self._views.clear()
        self.reset_draw_count = None
        for name in ("lap_idx", "lap_progress", "laps", "lap_ticks", "lap_start_ticks", "last_lap_ticks", "completed",
                     "hit_car", "contact"):
            setattr(self, name, None)
        for name in ("obs", "hits", "hit_points", "hit_seg", "hit_t", "reward", "fitness", "done", "crashed", "timed_out",
                     "nearest_idx", "pos_x", "pos_y", "rot", "speed", "act_throttle", "act_steer"):
            setattr(self, name, None)
        self.env.close()

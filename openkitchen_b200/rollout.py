"""Rollout collection for the policy-gradient trainers on top of ``BatchEnv`` (SURVEY.md section 8f, row N3).

The reference's PPO loop (RLRacers/PPO/ppo_sim.cpp:61-89, PPOAgent.hpp:68-102) builds one ``torch::tensor`` per agent
per tick, runs the actor on a batch of one, synchronises on ``.item<int>()`` for the sampled action and appends to
per-agent ``std::vector``s; the discounted returns are a host reverse scan (ExperienceBuffer.hpp:45-68).  Here the
whole rollout -- observation -> actor -> sample -> action table -> tick -> record, for every agent and ``steps`` ticks --
is captured once as ONE CUDA graph and replayed: no host work per tick, no launch latency between the ~10 small
kernels of a tick.  The returns are a batched reverse scan on the device.
"""
from __future__ import annotations

from typing import Callable

import torch

from .batch_env import BatchEnv


def discounted_returns(rewards: torch.Tensor, gamma: float = 0.99, done: torch.Tensor | None = None) -> torch.Tensor:
    """ExperienceBuffer::calculateDiscountedRewards (ExperienceBuffer.hpp:45-62) for every agent at once.

    rewards: f32[T, N] (one column per agent's ``saved_rewards``).  ret[t] = r[t] + gamma * ret[t + 1], scanned from the
    last tick backwards in binary32 with the reference's operation order.  ``done`` (u8/bool[T, N], optional) cuts the
    scan where an episode ended at tick t (the agent was reset afterwards), which the reference never needs because it
    rolls one episode per buffer."""
    if rewards.dim() != 2:
        raise ValueError("rewards must be [T, N]")
    out = torch.empty_like(rewards, dtype=torch.float32)
    acc = torch.zeros(rewards.shape[1], dtype=torch.float32, device=rewards.device)
    g = torch.tensor(gamma, dtype=torch.float32, device=rewards.device)
    for t in range(rewards.shape[0] - 1, -1, -1):
        if done is not None:
            acc = torch.where(done[t].bool(), torch.zeros_like(acc), acc)
        acc = rewards[t].to(torch.float32) + g * acc
        out[t] = acc
    return out


def discounted_returns_fused(env: BatchEnv, rewards: torch.Tensor, gamma: float = 0.99, done: torch.Tensor | None = None) -> torch.Tensor:
    """the same scan as ONE hand-written kernel (ok_discounted_returns: a thread per agent walks its column backwards)
    instead of 3 T torch launches; bit-identical to the loop above.  rewards f32[T, N] CUDA, done u8[T, N] or None."""
    if rewards.dim() != 2 or rewards.dtype != torch.float32 or not rewards.is_cuda:
        raise ValueError("rewards must be a CUDA f32[T, N] tensor")
    rewards = rewards.contiguous()
    out = torch.empty_like(rewards)
    d = None
    if done is not None:
        d = done.to(torch.uint8).contiguous()
    env.env.discounted_returns(rewards.data_ptr(), None if d is None else d.data_ptr(), out.data_ptr(), rewards.shape[0],
                               rewards.shape[1], float(gamma), env._stream())
    return out


def normalize_returns(returns: torch.Tensor) -> torch.Tensor:
    """(x - mean) / (std + eps) per agent (ExperienceBuffer.hpp:64-67: unbiased std, eps = FLT_EPSILON)"""
    eps = torch.finfo(torch.float32).eps
    return (returns - returns.mean(dim=0, keepdim=True)) / (returns.std(dim=0, keepdim=True) + eps)


class GraphedRollout:
    """``steps`` ticks of every agent as one CUDA graph.

    policy: obs f32[N, R] -> action probabilities f32[N, A] (a ``torch.nn.Module`` or any CUDA-graph-safe callable;
    its parameters may be updated in place between replays).  action_table: f32[A, 2] = (throttle, steering) per
    discrete action (kActionMap of the RL racers).  sample=False takes the argmax instead of sampling.
    After ``run()``: ``obs`` f32[T, N, R] (the state each action was chosen from), ``actions`` i64[T, N], ``log_prob``
    f32[T, N], ``rewards`` f32[T, N], ``dones`` u8[T, N] (after the tick).  With auto_reset and reset draws on
    (BatchEnv.set_reset_draws) the crashed agents restart at drawn points inside the graph, and each replay continues the
    reset stream.  With lap accounting on (BatchEnv.set_laps with a target) ``dones`` also marks the agents that completed
    their laps in that tick, and auto_reset restarts them too.  With races on (BatchEnv.set_races) every tick's race pass
    is captured with it: ``obs`` includes the other cars and ``dones`` the contact crashes."""

    def __init__(self, env: BatchEnv, policy: Callable[[torch.Tensor], torch.Tensor], action_table: torch.Tensor, steps: int,
                 sample: bool = True):
        self.env, self.policy, self.steps, self.sample = env, policy, int(steps), sample
        dev, n, r = env.device, env.n_agents, env.n_rays
        self.table = action_table.to(dev, torch.float32).contiguous()
        if self.table.dim() != 2 or self.table.shape[1] != 2:
            raise ValueError("action_table must be [A, 2] = (throttle, steering)")
        self.obs = torch.empty(self.steps, n, r, device=dev)
        self.actions = torch.empty(self.steps, n, dtype=torch.int64, device=dev)
        self.log_prob = torch.empty(self.steps, n, device=dev)
        self.rewards = torch.empty(self.steps, n, device=dev)
        self.dones = torch.empty(self.steps, n, dtype=torch.uint8, device=dev)
        self._thr = torch.empty(n, device=dev)
        self._steer = torch.empty(n, device=dev)
        self.graph: torch.cuda.CUDAGraph | None = None

    @torch.no_grad()
    def _tick(self, t: int):
        obs = self.env.obs
        self.obs[t].copy_(obs)
        probs = self.policy(obs)
        a = torch.multinomial(probs, 1)[:, 0] if self.sample else probs.argmax(dim=-1)
        self.actions[t].copy_(a)
        self.log_prob[t].copy_(torch.log(probs.gather(1, a[:, None])[:, 0]))
        torch.index_select(self.table[:, 0], 0, a, out=self._thr)
        torch.index_select(self.table[:, 1], 0, a, out=self._steer)
        self.env.step(self._thr, self._steer)
        self.rewards[t].copy_(self.env.reward)
        self.dones[t].copy_(self.env.done)

    def run_eager(self):
        """the same rollout launched tick by tick (what the graph replaces; also the capture warm-up)"""
        for t in range(self.steps):
            self._tick(t)
        return self

    def capture(self):
        dev = self.env.device
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            self._tick(0)  # warm-up outside the capture: lazy initialisation of the policy / cuBLAS workspaces
            torch.cuda.synchronize(dev)
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph, stream=side):
                self.run_eager()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        return self

    def run(self):
        """one rollout of ``steps`` ticks from the env's current state (captures the graph on first use)"""
        if self.graph is None:
            self.capture()
        self.graph.replay()
        return self


class FusedActorRollout:
    """The PPO racers' rollout with the policy step as ONE hand-written kernel per tick (ok_ppo_actor) instead of ~10
    torch kernels: observation -> Linear(R, H) -> relu -> Linear(H, A) -> softmax -> clamp -> sample -> log-prob ->
    kActionMap -> action buffers, plus the recording of obs / action / log-prob and of the previous tick's reward / done
    (RLRacers/PPO/PPOAgent.hpp:79-102, Actor.hpp:9-26, ppo_sim.cpp:61-89).  One launch per tick (the policy step is phase 0
    of the step kernel's tiles; ``one_launch=False``: two launches, actor then step), all ``steps`` ticks captured as one
    CUDA graph.

    l1, l2: ``torch.nn.Linear`` modules (the reference's ``Actor::l1`` / ``l2``); their parameters are read in place,
    so an optimizer step between rollouts is picked up by the next replay.  After ``run()``: ``obs`` f32[T, N, R],
    ``actions`` i32[T, N], ``log_prob`` f32[T, N], ``rewards`` f32[T, N], ``dones`` u8[T, N] (crashed, or with lap
    accounting on (BatchEnv.set_laps) completed).  With races on (BatchEnv.set_races) ok_ppo_actor_step enqueues the race
    pass after each tick, so the graph holds it: ``obs`` includes the other cars and ``dones`` the contact crashes."""

    def __init__(self, env: BatchEnv, l1: torch.nn.Linear, l2: torch.nn.Linear, action_table: torch.Tensor, steps: int,
                 sample: bool = True, seed: int = 0x0C17C4E2, one_launch: bool = True):
        from ._capi import OkActorIO

        self.env, self.steps, self.sample, self.seed = env, int(steps), sample, int(seed)
        # one_launch: the policy step runs as phase 0 of the step kernel's tiles (ok_ppo_actor_step) -- a tick of a few
        # thousand agents is latency, and two kernels pay it twice; False = the two launches (ok_ppo_actor, then the step)
        self.one_launch = bool(one_launch)
        dev, n, r = env.device, env.n_agents, env.n_rays
        for m in (l1, l2):
            if m.weight.device != dev or m.weight.dtype != torch.float32 or not m.weight.is_contiguous() or m.bias is None:
                raise ValueError("l1 / l2 must be float32 Linear layers with bias on the env's device")
        if l1.in_features != r or l2.in_features != l1.out_features or l2.out_features > 8:
            raise ValueError("actor shape must be Linear(rays, H) -> Linear(H, A), A <= 8")
        self.l1, self.l2 = l1, l2
        self.table = action_table.to(dev, torch.float32).contiguous()
        if self.table.shape != (l2.out_features, 2):
            raise ValueError("action_table must be [A, 2] = (throttle, steering)")
        self.obs = torch.empty(self.steps, n, r, device=dev)
        self.actions = torch.empty(self.steps, n, dtype=torch.int32, device=dev)
        self.log_prob = torch.empty(self.steps, n, device=dev)
        self.probs = torch.empty(self.steps, n, l2.out_features, device=dev)
        self.rewards = torch.empty(self.steps, n, device=dev)
        self.dones = torch.empty(self.steps, n, dtype=torch.uint8, device=dev)
        self.uniform: torch.Tensor | None = None  # f32[T, N] explicit draws (tests); None = the kernel's Philox stream
        self._io = OkActorIO
        self._tick0 = 0
        self.graph: torch.cuda.CUDAGraph | None = None

    def _io_for(self, t: int, act: bool = True):
        io = self._io()
        if act:
            io.d_w1, io.d_b1 = self.l1.weight.data_ptr(), self.l1.bias.data_ptr()
            io.d_w2, io.d_b2 = self.l2.weight.data_ptr(), self.l2.bias.data_ptr()
            io.hidden, io.n_actions = self.l1.out_features, self.l2.out_features
            io.d_action_table = self.table.data_ptr()
            io.d_uniform = None if self.uniform is None else self.uniform[t].data_ptr()
            io.greedy = 0 if self.sample else 1
            io.d_action, io.d_log_prob = self.actions[t].data_ptr(), self.log_prob[t].data_ptr()
            io.d_probs, io.d_obs = self.probs[t].data_ptr(), self.obs[t].data_ptr()
        if t > 0:
            io.d_prev_reward, io.d_prev_done = self.rewards[t - 1].data_ptr(), self.dones[t - 1].data_ptr()
        return io

    def _actor(self, t: int, act: bool = True):
        """the policy step alone (ok_ppo_actor): actions into the env's buffers, records of tick t"""
        self.env.env.ppo_actor(self._io_for(t, act), self._tick0 + t, self.seed, self.env._stream())

    def _tick(self, t: int):
        """policy step + the tick that consumes its actions"""
        if self.one_launch:
            self.env.env.ppo_actor_step(self._io_for(t), self._tick0 + t, self.seed, self.env._stream())
            self.env._step_count += 1
        else:
            self._actor(t)
            self.env.step()  # the actions the kernel left in the env's buffers

    def run_eager(self):
        for t in range(self.steps):
            self._tick(t)
        self._actor(self.steps, act=False)  # the last tick's reward / done
        return self

    def capture(self):
        dev = self.env.device
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            torch.cuda.synchronize(dev)
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph, stream=side):
                self.run_eager()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        return self

    def run(self):
        """one rollout of ``steps`` ticks from the env's current state (captures the graph on first use; a replay draws
        the same Philox action stream again unless ``uniform`` is refreshed by the caller).  Episode starts are another
        matter: with auto_reset and reset draws on (BatchEnv.set_reset_draws), each replay continues the reset stream,
        whose counters live on the device, so consecutive rollouts start their episodes at new draws"""
        if self.graph is None:
            self.capture()
        self.graph.replay()
        return self

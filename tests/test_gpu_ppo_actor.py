"""GPU: N3 -- the fused PPO actor kernel (ok_ppo_actor) against a torch float32 reference of the reference's Actor
(RLRacers/PPO/Actor.hpp:9-26) and PPOAgent::updateAction (PPOAgent.hpp:79-102), the rollout it drives against the CPU
ORACLE (not against the product itself), and the discounted-return kernel against ExperienceBuffer's loop."""
import numpy as np
import pytest
import torch

import openkitchen_b200 as ok
from openkitchen_b200.rollout import FusedActorRollout, discounted_returns, discounted_returns_fused
from oracle.api import Oracle, have_ref

pytestmark = pytest.mark.gpu
FAN = np.array([-70, -30, 0, 30, 70], dtype=np.float32)  # PPOAgent.hpp:57-61
TABLE = [[60.0, 0.0], [30.0, 5.0], [30.0, -5.0]]        # PPOAgent::kActionMap


def _actor(rays=5, hidden=128, actions=3, seed=0):
    torch.manual_seed(seed)
    l1, l2 = torch.nn.Linear(rays, hidden).cuda(), torch.nn.Linear(hidden, actions).cuda()
    return l1, l2


def _reference_probs(l1, l2, obs):
    """Actor::forward + the clamp of PPOAgent::updateAction, plain torch float32"""
    with torch.no_grad():
        x = torch.relu(torch.nn.functional.linear(obs, l1.weight, l1.bias))
        p = torch.softmax(torch.nn.functional.linear(x, l2.weight, l2.bias), dim=1)
        return torch.clamp(p, 1e-8, 1.0 - 1e-8)


@pytest.mark.parametrize("rays,hidden,actions", [(5, 128, 3), (32, 64, 5), (15, 30, 8)])
def test_fused_actor_matches_the_torch_reference(rays, hidden, actions):
    n = 3000
    fan = FAN if rays == 5 else rays
    env = ok.BatchEnv(["Monza", "Sepang"], n, rays=fan, auto_reset=1)
    env.step_random(25)
    l1, l2 = _actor(rays, hidden, actions)
    table = torch.randn(actions, 2, device="cuda")
    r = FusedActorRollout(env, l1, l2, table, steps=1, sample=True)
    r.uniform = torch.rand(1, n, device="cuda")
    r._actor(0)
    torch.cuda.synchronize()
    want = _reference_probs(l1, l2, env.obs)
    got = r.probs[0]
    # tolerance: the kernel accumulates in another order than cuBLAS and uses expf; probabilities agree to 2e-6 absolute
    assert torch.allclose(got, want, rtol=0, atol=2e-6), float((got - want).abs().max())
    assert torch.equal(r.obs[0], env.obs)
    # the choice is the inverse CDF of the kernel's OWN clamped probabilities at the given uniform draw -- exactly
    cum = torch.cumsum(got, dim=1)
    target = r.uniform[0] * got.sum(dim=1)
    mine = torch.minimum((target[:, None] >= cum).sum(dim=1), torch.tensor(actions - 1, device="cuda")).to(torch.int32)
    # (sequential float accumulation in the kernel vs cumsum: allow a draw that lands within 1e-6 of a boundary)
    near = ((target[:, None] - cum).abs() < 1e-6).any(dim=1)
    assert torch.equal(r.actions[0][~near], mine[~near]) and near.float().mean() < 1e-3
    a = r.actions[0].long()
    assert torch.allclose(r.log_prob[0], torch.log(got.gather(1, a[:, None])[:, 0]), rtol=1e-6, atol=1e-6)
    assert torch.equal(env.act_throttle, table[a, 0]) and torch.equal(env.act_steer, table[a, 1])
    # greedy = argmax
    g = FusedActorRollout(env, l1, l2, table, steps=1, sample=False)
    g._actor(0)
    torch.cuda.synchronize()
    clear = (want.topk(2, dim=1).values[:, 0] - want.topk(2, dim=1).values[:, 1]) > 1e-5
    assert torch.equal(g.actions[0][clear].long(), want.argmax(dim=1)[clear])


def test_philox_sampling_follows_the_probabilities():
    """without explicit draws the kernel samples from its Philox stream: over many agents that share one observation the
    action frequencies are the probabilities (torch::multinomial's distribution), and ticks / agents draw independently"""
    n = 200_000
    env = ok.BatchEnv(["Monza"], n, rays=FAN)
    env.cast_rays()  # every agent sits at the same pose: identical observations
    l1, l2 = _actor(seed=3)
    r = FusedActorRollout(env, l1, l2, torch.tensor(TABLE), steps=1)
    counts = torch.zeros(3, device="cuda")
    for t in range(3):
        r._tick0 = t
        r._actor(0)
        counts += torch.bincount(r.actions[0].long(), minlength=3).float()
    p = _reference_probs(l1, l2, env.obs[:1])[0]
    freq = counts / counts.sum()
    assert torch.allclose(freq, p / p.sum(), atol=4e-3), (freq, p)
    r._tick0 = 0
    r._actor(0)
    first = r.actions[0].clone()
    r._tick0 = 1
    r._actor(0)
    assert 0.2 < (first != r.actions[0]).float().mean() < 0.9  # another tick, another draw


@pytest.mark.parametrize("one_launch", [True, False])
@pytest.mark.parametrize("kind", ["port", "reference"])
def test_fused_rollout_replayed_through_the_oracle(kind, one_launch):
    """Config 4's loop (ppo_sim.cpp:61-89) as one CUDA graph of one launch per tick (the policy step as phase 0 of the step
    kernel's tiles, ok_ppo_actor_step) or two (ok_ppo_actor, then the step).  The recorded actions are replayed
    through the CPU oracle (kind = "reference": the reference's own Agent / RaceTrack objects): observations, rewards
    and done flags the rollout recorded must be the oracle's, bit for bit."""
    if kind == "reference" and not have_ref():
        pytest.skip("oracle/_ref/libokref.so not built")
    n, steps = 192, 60
    env = ok.BatchEnv(["Monza", "Spielberg"], n, rays=FAN, reward_mode=ok.REWARD_CONSTANT, auto_reset=1)
    ora = Oracle(kind, movement_mode=0, reward_mode=3, auto_reset=1)
    for nm in ("Monza", "Spielberg"):
        ora.add_track(ok.track_columns(nm))
    tid = (np.arange(n) * 2 // n).astype(np.int32)
    ora.alloc_agents(n, FAN, tid)
    pts = (np.arange(n) * 37 % 700).astype(np.int32)
    env.reset(None, torch.from_numpy(pts).cuda())
    ora.reset(None, pts)
    env.cast_rays()  # the initial observation (ppo_sim.cpp:56-57 steps once with a zero action; a cast is the same lidar)
    ora.cast_rays()
    l1, l2 = _actor(seed=1)
    table = torch.tensor(TABLE, device="cuda")
    r = FusedActorRollout(env, l1, l2, table, steps=steps, sample=True, one_launch=one_launch)
    r.run()
    torch.cuda.synchronize()
    acts = r.actions.cpu().numpy()
    tab = np.asarray(TABLE, dtype=np.float32)
    assert len(np.unique(acts)) == 3
    for t in range(steps):
        assert np.array_equal(r.obs[t].cpu().numpy().view(np.uint32), ora.buffer("obs").view(np.uint32)), f"obs at tick {t}"
        ora.step(tab[acts[t], 0], tab[acts[t], 1])
        assert np.array_equal(r.rewards[t].cpu().numpy(), ora.buffer("reward")), f"reward at tick {t}"
        assert np.array_equal(r.dones[t].cpu().numpy(), ora.buffer("done")), f"done at tick {t}"
    assert r.dones.sum() > 0, "nobody crashed: the rollout is too short to exercise the auto-reset"
    for name in ("pos_x", "pos_y", "rot", "crashed"):
        assert np.array_equal(env[name].cpu().numpy().view(np.uint8), ora.buffer(name).view(np.uint8)), name
    # a second replay continues from the current state and records the same kind of data
    r.run()
    torch.cuda.synchronize()
    assert torch.isfinite(r.log_prob).all() and (r.log_prob <= 0).all()


def test_discounted_return_kernel_is_the_reference_loop():
    """ExperienceBuffer::calculateDiscountedRewards (ExperienceBuffer.hpp:45-62), one agent's loop in binary32"""
    rng = np.random.default_rng(0)
    t_steps, n = 300, 513
    rew = rng.normal(size=(t_steps, n)).astype(np.float32)
    rew[:, 0] = 1.0  # ppo_sim.cpp:76
    done = (rng.random((t_steps, n)) < 0.02).astype(np.uint8)
    env = ok.BatchEnv(["Monza"], 4, rays=FAN)
    for use_done in (False, True):
        got = discounted_returns_fused(env, torch.from_numpy(rew).cuda(), 0.99, torch.from_numpy(done).cuda() if use_done else None)
        got = got.cpu().numpy()
        for a in (0, 1, 7, n - 1):
            cum, want = np.float32(0.0), np.zeros(t_steps, dtype=np.float32)
            for i in range(t_steps - 1, -1, -1):
                if use_done and done[i, a]:
                    cum = np.float32(0.0)
                cum = np.float32(rew[i, a] + np.float32(np.float32(0.99) * cum))
                want[i] = cum
            assert np.array_equal(got[:, a].view(np.uint32), want.view(np.uint32)), (use_done, a)
        ref = discounted_returns(torch.from_numpy(rew).cuda(), 0.99, torch.from_numpy(done).cuda() if use_done else None)
        assert torch.equal(torch.from_numpy(got).cuda(), ref)


@pytest.mark.parametrize("kernel,n", [("staged", 4096), ("unstaged", 700)])
def test_one_launch_tick_equals_the_two_launches(monkeypatch, kernel, n):
    """ok_ppo_actor_step (policy step fused into the step kernel) against ok_ppo_actor + ok_launch_step on twin envs: every
    rollout record and every env buffer, bit for bit, in the beam kernel shape that has a fused instantiation (unstaged) and
    in those that fall back to the two launches."""
    monkeypatch.setenv("OK_BEAM_KERNEL", kernel)
    l1, l2 = _actor(seed=3)
    table = torch.tensor(TABLE, device="cuda")
    outs = []
    for one_launch in (True, False):
        env = ok.BatchEnv(["Monza", "Zandvoort"], n, rays=FAN, reward_mode=ok.REWARD_CONSTANT, auto_reset=1)
        pts = (np.arange(n) * 53 % 600).astype(np.int32)
        env.reset(None, torch.from_numpy(pts).cuda())
        env.cast_rays()
        r = FusedActorRollout(env, l1, l2, table, steps=40, sample=True, one_launch=one_launch)
        before = env.env.launch_stats().kernel_launches
        r.run_eager()
        launched = env.env.launch_stats().kernel_launches - before
        # 40 ticks + the record of the last tick's reward / done: one launch per tick where a fused instantiation exists
        assert launched == (41 if one_launch and kernel == "unstaged" else 81), launched
        env.reset(None, torch.from_numpy(pts).cuda())
        env.cast_rays()
        r.run()
        torch.cuda.synchronize()
        outs.append((r, env))
    (a, ea), (b, eb) = outs
    for name in ("obs", "actions", "log_prob", "probs", "rewards", "dones"):
        assert torch.equal(getattr(a, name), getattr(b, name)), name
    assert a.dones.sum() > 0
    for name in ok.BUFFERS:
        assert np.array_equal(ea.env.read(name).view(np.uint8), eb.env.read(name).view(np.uint8)), name

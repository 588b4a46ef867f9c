"""GPU: reset draws (OkResetDraws).  The drawn auto-reset inside every step kernel and the explicit drawn reset against the
port oracle with the draws of tests/reset_draws_oracle.py, bit for bit on every buffer and on the counters; the fused actor + tick; CUDA graphs whose replays continue
the reset stream; sharding; and the self-check count of the kernels that ran."""
import numpy as np
import pytest
import torch

import openkitchen_b200 as ok
from openkitchen_b200.dlpack import DeviceBuffer
from tests.reset_draws_oracle import STARTING_IDX, DrawnResets, draw
from tests.util import ALL_BUFS, assert_same, make_pair, spread_points

pytestmark = pytest.mark.gpu

SEED = 0x5EED


def counts(env) -> np.ndarray:
    """host copy of the env's reset-draw counters"""
    env.sync()
    return torch.from_dlpack(DeviceBuffer(env, "k", env.reset_draw_counts_info())).view(torch.int32).cpu().numpy().view(np.uint32).copy()


def no_violations(env):
    n, _ = env.debug_violations()
    assert n == 0, f"{n} out-of-range indices counted"


def run_pair(flags, mode=ok.MOVE_VELOCITY, raycast=ok.RAYCAST_BEAM, n=96, rays=16, ticks=300, names=None, **cfg):
    names = names or ["Monza", "Spa", "Silverstone", "Austin"]
    env, ora, tid = make_pair(names, n, rays, movement_mode=mode, raycast_mode=raycast,
                              reward_mode=ok.REWARD_CMAES_PROGRESS, auto_reset=1, **cfg)
    env.set_reset_draw_flags(SEED, flags)
    drawn = DrawnResets(ora, SEED, flags)
    pts = spread_points(ora, tid)
    env.reset(None, pts)
    ora.reset(None, pts)
    for step in range(ticks):
        env.launch_steps_random(step, 1)
        ora.fill_random_actions(step)
        drawn.step()
        if step % 50 == 49:
            assert_same(env, ora, ctx=f"flags {flags} tick {step}")
            assert np.array_equal(counts(env), drawn.k), f"counters, tick {step}"
    k = counts(env)
    if flags:
        assert k.sum() >= n, "too few drawn resets for the test to mean anything"
    else:
        assert not k.any()
    no_violations(env)
    return env, ora


@pytest.mark.parametrize("flags", range(8))
def test_every_flag_combination_matches_the_oracle(flags):
    run_pair(flags)


@pytest.mark.parametrize("raycast", [ok.RAYCAST_GRID, ok.RAYCAST_BRUTE])
@pytest.mark.parametrize("flags", [5, 7])
def test_grid_and_brute_modes(raycast, flags):
    run_pair(flags, raycast=raycast, n=64, ticks=300)


def test_acceleration_mode():
    run_pair(7, mode=ok.MOVE_ACCELERATION, ticks=300)


@pytest.mark.parametrize("kernel", ["staged", "unstaged"])
def test_both_beam_kernel_shapes(kernel, monkeypatch):
    """the staged kernel (populations from 65,536 rays per tick) and the unstaged one, forced at a size the oracle can follow"""
    monkeypatch.setenv("OK_BEAM_KERNEL", kernel)
    env, _ = run_pair(7, n=160, ticks=300)
    staged_block = env.launch_stats().block_threads
    assert (staged_block == 1024) == (kernel == "staged"), staged_block


def test_natural_staged_population():
    """a population above the staged threshold, as the sizing picks it: device against oracle on a slice of the run"""
    env, ora, tid = make_pair(["Monza", "Spa"], 2304, 32, reward_mode=ok.REWARD_CMAES_PROGRESS, auto_reset=1)
    assert env.launch_stats().block_threads == 1024, "not the staged shape"
    env.set_reset_draws(SEED, point=True, lane=True, heading=True)
    drawn = DrawnResets(ora, SEED, 7)
    pts = spread_points(ora, tid)
    env.reset(None, pts)
    ora.reset(None, pts)
    for step in range(100):
        env.launch_steps_random(step, 1)
        ora.fill_random_actions(step)
        drawn.step()
    assert_same(env, ora, ctx="staged population")
    assert np.array_equal(counts(env), drawn.k) and counts(env).sum() > 0
    no_violations(env)


def _twin_reset_args(env, idx, flags, k):
    """(pt, alpha, off) of the drawn reset of agents idx at counters k, by the definition"""
    tid = env.read("track_id")
    n_pts = np.array([env.track_info(int(tid[a])).n_points for a in idx], dtype=np.int64)
    pt, alpha, off = draw(SEED, flags, np.asarray(idx, np.uint64), k[idx], n_pts, np.minimum(STARTING_IDX, n_pts - 1))
    return pt, (alpha if flags & 2 else None), off


@pytest.mark.parametrize("how", ["indices", "mask", "all"])
@pytest.mark.parametrize("flags", [0, 3, 7])
def test_explicit_drawn_reset_equals_ok_reset_agents(how, flags):
    names, n = ["Monza", "Spa"], 50
    a, _, tid = make_pair(names, n, 9, reward_mode=ok.REWARD_CMAES_PROGRESS)
    b, _, _ = make_pair(names, n, 9, reward_mode=ok.REWARD_CMAES_PROGRESS)
    for e in (a, b):
        e.set_reset_draw_flags(SEED, flags)
        e.launch_steps_random(0, 7)
    rng = np.random.default_rng(3)
    mask = (rng.random(n) < 0.4).astype(np.uint8)
    for rnd in range(3):  # the counters advance: three rounds draw three different resets
        k = counts(a)
        idx = {"indices": np.flatnonzero(mask)[::-1].copy(), "mask": np.flatnonzero(mask), "all": np.arange(n)}[how]
        before = {nm: a.read(nm) for nm in ALL_BUFS}
        if how == "indices":
            a.reset_drawn(agent_idx=idx)
        elif how == "mask":
            a.reset_drawn(mask=mask)
        else:
            a.reset_drawn()
        pt, la, ho = _twin_reset_args(b, idx, flags, k)
        b.reset(idx, pt, la, ho)
        for nm in ALL_BUFS:
            assert np.array_equal(a.read(nm).view(np.uint8), b.read(nm).view(np.uint8)), (nm, rnd)
        k2 = counts(a)
        touched = np.zeros(n, bool)
        touched[idx] = True
        assert np.array_equal(k2 - k, touched.astype(np.uint32))
        for nm in ("pos_x", "pos_y", "rot", "reset_pt", "start_x"):  # an unmasked agent keeps its state
            assert np.array_equal(a.read(nm)[~touched].view(np.uint8), before[nm][~touched].view(np.uint8)), nm
    no_violations(a)


def _actor(env, hidden=16, n_actions=5, seed=0):
    g = torch.Generator().manual_seed(seed)
    l1 = torch.nn.Linear(env.n_rays, hidden)
    l2 = torch.nn.Linear(hidden, n_actions)
    with torch.no_grad():
        for m in (l1, l2):
            m.weight.copy_(torch.randn(m.weight.shape, generator=g) * 0.5)
            m.bias.copy_(torch.randn(m.bias.shape, generator=g) * 0.1)
    table = torch.tensor([[0.0, 0.0], [80.0, 0.0], [80.0, 4.0], [80.0, -4.0], [40.0, 2.0]])[:n_actions]
    return l1.to(env.device), l2.to(env.device), table


def _batch(n=128, rays=5, auto_reset=1, **cfg):
    return ok.BatchEnv(["Monza", "Spa"], n, rays=rays, reward_mode=ok.REWARD_CONSTANT, auto_reset=auto_reset, **cfg)


def _same_envs(a, b, ctx):
    for nm in ok.BUFFERS:
        assert torch.equal(a[nm].view(torch.uint8), b[nm].view(torch.uint8)), (nm, ctx)
    assert torch.equal(a.reset_draw_count.view(torch.int32), b.reset_draw_count.view(torch.int32)), ctx


def test_fused_actor_step_equals_actor_plus_step():
    from openkitchen_b200.rollout import FusedActorRollout

    a, b = _batch(), _batch()
    for e in (a, b):
        e.set_reset_draws(SEED, point=True, lane=True, heading=True)
    l1, l2, table = _actor(a)
    ra = FusedActorRollout(a, l1, l2, table, 200, one_launch=True).run_eager()
    rb = FusedActorRollout(b, l1, l2, table, 200, one_launch=False).run_eager()
    torch.cuda.synchronize()
    _same_envs(a, b, "fused vs two launches")
    assert torch.equal(ra.actions, rb.actions) and torch.equal(ra.dones, rb.dones)
    assert int(a.reset_draw_count.view(torch.int32).to(torch.int64).sum()) > a.n_agents // 2


def test_graph_replays_continue_the_reset_stream():
    from openkitchen_b200.rollout import FusedActorRollout

    a, b = _batch(), _batch()
    for e in (a, b):
        e.set_reset_draws(SEED, point=True, lane=True, heading=True)
    l1, l2, table = _actor(a)
    ra = FusedActorRollout(a, l1, l2, table, 60)
    rb = FusedActorRollout(b, l1, l2, table, 60)
    ra.run()
    torch.cuda.synchronize()
    start1 = torch.stack([a["start_x"], a["start_y"]]).clone()
    k1 = a.reset_draw_count.view(torch.int32).to(torch.int64).clone()
    ra.run()
    torch.cuda.synchronize()
    rb.run_eager()
    rb.run_eager()
    torch.cuda.synchronize()
    _same_envs(a, b, "two replays vs 2T eager ticks")
    k2 = a.reset_draw_count.view(torch.int32).to(torch.int64)
    assert int(k1.sum()) > 0 and bool((k2 > k1).any()), "the second replay made no drawn reset"
    again = (k2 > k1)
    assert not torch.equal(torch.stack([a["start_x"], a["start_y"]])[:, again], start1[:, again])


def test_reset_drawn_of_done_captures_into_a_graph():
    """env.reset_drawn(env.done) inside a CUDA graph (a host synchronisation would fail the capture): the replays equal the
    same calls made eagerly on a twin.  The graph keeps the tick numbers of its capture (0..4), so the twin uses those."""
    a, c = _batch(auto_reset=0), _batch(auto_reset=0)
    for e in (a, c):
        e.set_reset_draws(SEED, point=True, lane=False, heading=True)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(g, stream=side):
            for _ in range(5):
                a.step_random(1)
                a.reset_drawn(a.done)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    resets = 0
    for _ in range(20):
        g.replay()
        for t in range(5):
            c.env.launch_steps_random(t, 1, stream=c._stream())
            resets += int(c.done.sum())
            c.reset_drawn(c.done)
    torch.cuda.synchronize()
    assert resets > 0
    _same_envs(a, c, "graph replays vs eager")
    assert int(a.reset_draw_count.view(torch.int32).to(torch.int64).sum()) == resets


def test_index_reset_on_the_device():
    a, b = _batch(), _batch()
    for e in (a, b):
        e.set_reset_draws(SEED, point=True, lane=True, heading=True)
        e.step_random(40)
    idx = torch.tensor([5, 0, 77, 31], device=a.device)
    a.reset_drawn(idx)
    b.env.reset_drawn(agent_idx=idx.cpu().numpy())
    torch.cuda.synchronize()
    _same_envs(a, b, "device indices vs host indices")


def test_shard_reproduces_its_slice():
    names = ["Monza", "Spa", "Silverstone"]
    n, lo = 120, 48
    fan = ok.ray_fan(9)
    tid = (np.arange(n) % len(names)).astype(np.int32)

    def env_for(base, t):
        e = ok.Env(device=0, reward_mode=ok.REWARD_CMAES_PROGRESS, auto_reset=1, agent_id_base=base)
        for nm in names:
            e.add_named_track(nm)
        e.alloc_agents(len(t), fan, t)
        e.set_reset_draws(SEED, point=True, lane=True, heading=True)
        return e

    full, shard = env_for(0, tid), env_for(lo, tid[lo:])
    for e in (full, shard):
        e.launch_steps_random(0, 250)
    k = counts(full)
    assert k.sum() > n
    assert np.array_equal(k[lo:], counts(shard))
    for nm in ALL_BUFS:
        assert np.array_equal(full.read(nm)[lo:].view(np.uint8), shard.read(nm).view(np.uint8)), nm


def test_draws_off_by_default_and_settable():
    env, _, _ = make_pair(["Monza"], 8, 5)
    assert env.reset_draws() == {"seed": 0, "point": False, "lane": False, "heading": False}
    env.set_reset_draws(7, point=False, lane=True)
    assert env.reset_draws() == {"seed": 7, "point": False, "lane": True, "heading": False}
    with pytest.raises(ok.OkError):
        import ctypes as C

        from openkitchen_b200 import _capi

        d = _capi.OkResetDraws(seed=1, flags=16)
        _capi.check(env.lib.ok_set_reset_draws(env.h, C.byref(d)))
    before = env.launch_stats().kernel_launches
    env.reset_drawn()
    assert env.launch_stats().kernel_launches == before + 1

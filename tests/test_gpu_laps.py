"""GPU: lap accounting (OkLaps).  Every step kernel shape against the port oracle with the accounting of
tests/laps_oracle.py, bit for bit on every buffer and on the seven lap arrays, with near-complete state planted so that
completions, lap times, completed-agent auto-resets and reversals happen within a few hundred ticks; the fused actor +
tick; real laps driven by a centre-line follower; CUDA graphs whose replays continue the state; accounting off; the
host done mirror; and the self-check count of the kernels that ran."""
import numpy as np
import pytest
import torch

import openkitchen_b200 as ok
from openkitchen_b200.dlpack import DeviceBuffer
from tests.laps_oracle import FIELDS, Laps, lap_rule
from tests.reset_draws_oracle import DrawnResets
from tests.util import assert_same, make_pair, spread_points

pytestmark = pytest.mark.gpu

SEED = 0x1A95


def lap_views(env) -> dict:
    """torch views of an Env's seven lap arrays"""
    return {f: torch.from_dlpack(DeviceBuffer(env, f, info)) for f, info in env.lap_buffers_info().items()}


def read_laps(env) -> dict:
    env.sync()
    out = {}
    for f, v in lap_views(env).items():
        t = v.view(torch.int32) if v.element_size() == 4 else v
        out[f] = t.cpu().numpy().view(FIELDS[f]).copy()
    return out


def write_laps(env, s: dict):
    env.sync()
    for f, v in lap_views(env).items():
        a = torch.from_numpy(np.ascontiguousarray(s[f]).view(np.int32 if v.element_size() == 4 else np.uint8).copy())
        (v.view(torch.int32) if v.element_size() == 4 else v).copy_(a.to(v.device))
    torch.cuda.synchronize()


def assert_laps(env, laps: Laps, ctx):
    got = read_laps(env)
    for f in FIELDS:
        bad = np.flatnonzero(got[f] != laps.s[f])
        assert bad.size == 0, f"{ctx}: lap array {f}: {bad.size} mismatches, first agent {bad[0]}: gpu={got[f][bad[0]]} oracle={laps.s[f][bad[0]]}"


def no_violations(env):
    n, _ = env.debug_violations()
    assert n == 0, f"{n} out-of-range indices counted"


def plant(laps: Laps, env, rng, frac=0.5):
    """near-complete state on a random subset of agents: progress a few points below k*P with laps = k - 1, so a lap
    completes within a few ticks of forward driving (and a reversal keeps it from completing), the same in both"""
    s = laps.s
    pick = np.flatnonzero(rng.random(laps.ora.n) < frac)
    k = rng.integers(1, 3, pick.size)
    s["laps"][pick] = (k - 1).astype(np.int32)
    s["progress"][pick] = (k * laps.n_points[pick] - rng.integers(0, 6, pick.size)).astype(np.int32)
    s["ticks"][pick] = rng.integers(50, 500, pick.size).astype(np.uint32)
    s["lap_start"][pick] = (s["ticks"][pick] - rng.integers(0, 40, pick.size)).astype(np.uint32)
    write_laps(env, s)


def run_pair(mode=ok.MOVE_VELOCITY, raycast=ok.RAYCAST_BEAM, reward=ok.REWARD_CONSTANT, draws=0, auto_reset=1, target=2,
             n=160, rays=16, ticks=300, names=None, check_every=50):
    names = names or ["Monza", "Spa", "Silverstone", "Austin"]
    env, ora, tid = make_pair(names, n, rays, movement_mode=mode, raycast_mode=raycast, reward_mode=reward,
                              auto_reset=auto_reset)
    env.set_reset_draw_flags(SEED, draws)
    drawn = DrawnResets(ora, SEED, draws)
    laps = Laps(ora, drawn)
    pts = spread_points(ora, tid)
    env.reset(None, pts)
    laps.reset(None, pts)
    env.set_laps(target)
    laps.set(True, target)
    assert_laps(env, laps, "after set_laps")
    plant(laps, env, np.random.default_rng(n + ticks + draws))
    completions = lap_events = 0
    for step in range(ticks):
        env.launch_steps_random(step, 1)
        ora.fill_random_actions(step)
        before = laps.s["laps"].copy()
        laps.step()
        lap_events += int(np.sum(laps.s["laps"] > before))  # a restarted agent cannot complete a lap in its first tick
        completions += int(laps.s["completed"].sum())
        if step % check_every == check_every - 1 or step == ticks - 1:
            assert_same(env, ora, ctx=f"tick {step}")
            assert_laps(env, laps, f"tick {step}")
    assert lap_events >= n // 10, "too few laps for the test to mean anything"
    if target:
        assert completions > 0
    no_violations(env)
    return env, ora, laps


@pytest.mark.parametrize("auto_reset", [0, 1])
@pytest.mark.parametrize("draws", [0, 7])
@pytest.mark.parametrize("kernel", ["staged", "unstaged"])
def test_beam_kernel_shapes_match_the_oracle(kernel, draws, auto_reset, monkeypatch):
    """the staged and the unstaged beam kernel, forced at a size the oracle can follow; draws off and on, auto_reset off
    and on; a reward mode that does not search the centre line without accounting (constant) and one that does"""
    monkeypatch.setenv("OK_BEAM_KERNEL", kernel)
    reward = ok.REWARD_CONSTANT if kernel == "staged" else ok.REWARD_CMAES_PROGRESS
    env, _, laps = run_pair(reward=reward, draws=draws, auto_reset=auto_reset)
    assert (env.launch_stats().block_threads == 1024) == (kernel == "staged")
    if draws and auto_reset:
        assert laps.drawn.k.sum() > 0


@pytest.mark.parametrize("raycast", [ok.RAYCAST_GRID, ok.RAYCAST_BRUTE])
@pytest.mark.parametrize("draws", [0, 5])
def test_grid_and_brute_modes(raycast, draws):
    run_pair(raycast=raycast, draws=draws, reward=ok.REWARD_Q_PROGRESS, n=64, ticks=250)


@pytest.mark.parametrize("reward", [ok.REWARD_MIN_RAY, ok.REWARD_TRACK_INDEX])
def test_acceleration_mode(reward):
    run_pair(mode=ok.MOVE_ACCELERATION, reward=reward, draws=7, ticks=300)


def test_natural_staged_population():
    """a population above the staged threshold, as the sizing picks it, against the oracle on a slice of the run"""
    env, ora, tid = make_pair(["Monza", "Spa"], 2304, 32, reward_mode=ok.REWARD_DISPLACEMENT, auto_reset=1)
    assert env.launch_stats().block_threads == 1024, "not the staged shape"
    env.set_reset_draws(SEED, point=True, lane=True, heading=True)
    laps = Laps(ora, DrawnResets(ora, SEED, 7))
    pts = spread_points(ora, tid)
    env.reset(None, pts)
    laps.reset(None, pts)
    env.set_laps(1)
    laps.set(True, 1)
    plant(laps, env, np.random.default_rng(5))
    lap_events = 0
    for step in range(80):
        env.launch_steps_random(step, 1)
        ora.fill_random_actions(step)
        before = laps.s["laps"].copy()
        laps.step()
        lap_events += int(np.sum(laps.s["laps"] > before))
    assert_same(env, ora, ctx="staged population")
    assert_laps(env, laps, "staged population")
    assert lap_events > 0
    no_violations(env)


def test_explicit_resets_restart_the_lap_state():
    env, ora, tid = make_pair(["Monza", "Spa"], 48, 9, reward_mode=ok.REWARD_CONSTANT)
    env.set_laps(0)
    laps = Laps(ora)
    laps.set(True, 0)
    for step in range(40):
        env.launch_steps_random(step, 1)
        ora.fill_random_actions(step)
        laps.step()
    idx = np.array([3, 17, 40])
    env.reset(idx, np.array([10, 20, 30]))
    laps.reset(idx, np.array([10, 20, 30]))
    assert_laps(env, laps, "after ok_reset_agents")
    assert not read_laps(env)["ticks"][idx].any() and read_laps(env)["ticks"].max() > 0
    env.reset_drawn(agent_idx=[5])
    got = read_laps(env)
    assert got["ticks"][5] == 0 and got["lap_idx"][5] == env.read("prev_idx")[5]
    no_violations(env)


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


LAP_VIEWS = ("lap_idx", "lap_progress", "laps", "lap_ticks", "lap_start_ticks", "last_lap_ticks", "completed")


def _batch(n=128, rays=5, auto_reset=1, **cfg):
    return ok.BatchEnv(["Monza", "Spa"], n, rays=rays, reward_mode=ok.REWARD_CONSTANT, auto_reset=auto_reset, **cfg)


def _plant_batch(env, seed=1):
    """progress a few points below P on every other agent"""
    P = torch.tensor(env.points_per_track, device=env.device)[env.track_id.to(env.device).long()].to(torch.int32)
    g = torch.Generator(device="cpu").manual_seed(seed)
    short = torch.randint(0, 4, (env.n_agents,), generator=g).to(env.device, torch.int32)
    every_other = torch.arange(env.n_agents, device=env.device) % 2 == 0
    env.lap_progress.copy_(torch.where(every_other, P - short, env.lap_progress))


def _same_envs(a, b, ctx):
    for nm in ok.BUFFERS:
        assert torch.equal(a[nm].view(torch.uint8), b[nm].view(torch.uint8)), (nm, ctx)
    for nm in LAP_VIEWS:
        assert torch.equal(getattr(a, nm).view(torch.uint8), getattr(b, nm).view(torch.uint8)), (nm, ctx)


@pytest.mark.parametrize("draws", [False, True])
def test_fused_actor_step_equals_actor_plus_step(draws):
    from openkitchen_b200.rollout import FusedActorRollout

    a, b = _batch(), _batch()
    for e in (a, b):
        if draws:
            e.set_reset_draws(SEED, point=True, lane=True, heading=True)
        e.set_laps(1)
        _plant_batch(e)
    l1, l2, table = _actor(a)
    ra = FusedActorRollout(a, l1, l2, table, 200, one_launch=True).run_eager()
    rb = FusedActorRollout(b, l1, l2, table, 200, one_launch=False).run_eager()
    torch.cuda.synchronize()
    _same_envs(a, b, "fused vs two launches")
    assert torch.equal(ra.actions, rb.actions) and torch.equal(ra.dones, rb.dones)
    assert int(ra.dones.sum()) > 0 and int(a.lap_ticks.view(torch.int32).to(torch.int64).sum()) > 0


def test_graph_with_reset_drawn_of_done_continues_the_lap_state():
    """env.reset_drawn(env.done) and lap accounting inside a CUDA graph: its replays equal the same calls made eagerly on
    a twin, and the lap state carries on from one replay to the next.  The graph keeps the tick numbers of its capture
    (0..4), so the twin uses those."""
    a, c = _batch(auto_reset=0), _batch(auto_reset=0)
    for e in (a, c):
        e.set_reset_draws(SEED, point=True, lane=False, heading=True)
        e.set_laps(1)
        _plant_batch(e)
    torch.cuda.synchronize()
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
    completions, ticks_seen = 0, []
    for _ in range(20):
        g.replay()
        for t in range(5):
            c.env.launch_steps_random(t, 1, stream=c._stream())
            completions += int(c.completed.sum())
            c.reset_drawn(c.done)
        torch.cuda.synchronize()
        ticks_seen.append(int(a.lap_ticks.view(torch.int32).to(torch.int64).max()))
    assert completions > 0
    _same_envs(a, c, "graph replays vs eager")
    assert max(ticks_seen) > 5, "the lap state did not carry over from one replay to the next"


def test_accounting_off_leaves_the_arrays_alone():
    env, ora, tid = make_pair(["Monza", "Spa"], 64, 9, reward_mode=ok.REWARD_CONSTANT, auto_reset=1)
    assert env.laps() == {"enabled": False, "target": 0}
    rng = np.random.default_rng(2)
    junk = {f: rng.integers(0, 200, 64).astype(dt) for f, dt in FIELDS.items()}
    junk["completed"][:] = 1
    write_laps(env, junk)
    for step in range(200):
        env.launch_steps_random(step, 1)
        ora.fill_random_actions(step)
        ora.step()
    assert_same(env, ora, ctx="accounting off")
    got = read_laps(env)
    for f in FIELDS:
        assert np.array_equal(got[f], junk[f]), f
    assert np.array_equal(env.read("done"), env.read("crashed"))
    # on, then off: the state stays where the last tick with accounting on left it
    env.set_laps(0)
    env.launch_steps_random(1000, 3)
    on = read_laps(env)
    assert np.all(on["completed"] == 0) and on["ticks"].max() <= 3
    env.set_laps(0, enabled=False)
    env.launch_steps_random(2000, 5)
    off = read_laps(env)
    for f in FIELDS:
        assert np.array_equal(off[f], on[f]), f
    env.cast_rays()
    for f, v in read_laps(env).items():
        assert np.array_equal(v, on[f]), f
    no_violations(env)


def test_switching_on_restarts_every_agent_at_its_pose():
    env, ora, tid = make_pair(["Monza", "Spa"], 64, 9, reward_mode=ok.REWARD_CONSTANT)
    env.launch_steps_random(0, 30)
    write_laps(env, {f: np.full(64, 7, dt) for f, dt in FIELDS.items()})
    env.set_laps(3)
    assert env.laps() == {"enabled": True, "target": 3}
    got = read_laps(env)
    x, y = env.read("pos_x"), env.read("pos_y")
    want, _, _ = env.track_query(x, y, env.read("track_id"))
    assert np.array_equal(got["lap_idx"], want)
    for f in FIELDS:
        if f != "lap_idx":
            assert not got[f].any(), f
    write_laps(env, {f: np.full(64, 7, dt) for f, dt in FIELDS.items()})
    env.set_laps(5)  # on -> on: no restart
    assert read_laps(env)["ticks"][0] == 7


def test_host_done_mirror_includes_completions():
    env, ora, tid = make_pair(["Monza"], 32, 9, reward_mode=ok.REWARD_CONSTANT)
    env.set_laps(1)
    s = read_laps(env)
    P = env.track_info(0).n_points
    s["progress"][:16] = P - 1
    write_laps(env, s)
    done = np.zeros(32, np.uint8)
    thr = np.full(32, 60.0, np.float32)
    steer = np.zeros(32, np.float32)
    for _ in range(30):
        env.step_host(thr, steer, None, None, done)
        assert np.array_equal(done, env.read("done"))
    got = read_laps(env)
    assert got["completed"][:16].sum() > 0
    assert np.array_equal(done, (env.read("crashed") | got["completed"]).astype(np.uint8))


def test_real_laps_on_a_short_track():
    """A centre-line follower drives real laps of Oschersleben (739 points); laps and last_lap agree with a host recount
    from the nearest_idx recorded every tick."""
    n, ticks, speed, ahead = 64, 2400, 300.0, 6
    env = ok.BatchEnv(["Oschersleben"], n, rays=9, reward_mode=ok.REWARD_CONSTANT)
    P = env.points_per_track[0]
    assert P == 739
    start = torch.arange(n, device=env.device, dtype=torch.int32) * P // n
    env.reset(None, start)
    env.set_laps(0)
    cx = torch.from_numpy(env.env.track_array(0, "x")).to(env.device)
    cy = torch.from_numpy(env.env.track_array(0, "y")).to(env.device)
    lap_idx0 = env.lap_idx.clone()
    thr = torch.full((n,), speed, device=env.device)
    hist = torch.empty(ticks, n, dtype=torch.int32, device=env.device)
    for t in range(ticks):
        tgt = (env.nearest_idx.long() + ahead) % P
        want = torch.rad2deg(torch.atan2(cy[tgt] - env.pos_y, cx[tgt] - env.pos_x))
        steer = torch.clamp(torch.remainder(want - env.rot + 180.0, 360.0) - 180.0, -10.0, 10.0)
        env.step(thr, steer)
        hist[t].copy_(env.nearest_idx)
    torch.cuda.synchronize()
    assert not env.crashed.any(), "the follower crashed"
    h = hist.cpu().numpy()
    s = {f: np.zeros(n, dtype=dt) for f, dt in FIELDS.items()}
    s["lap_idx"] = lap_idx0.cpu().numpy()
    for t in range(ticks):
        s = lap_rule(s, h[t], P, 0, np.ones(n, bool))
    got = {"laps": env.laps.cpu().numpy(), "last_lap": env.last_lap_ticks.view(torch.int32).cpu().numpy().view(np.uint32),
           "progress": env.lap_progress.cpu().numpy(), "ticks": env.lap_ticks.view(torch.int32).cpu().numpy().view(np.uint32)}
    for f, v in got.items():
        assert np.array_equal(v, s[f]), f
    assert np.all(s["laps"] >= 2) and np.all(s["ticks"] == ticks)
    assert np.all((s["last_lap"] > 600) & (s["last_lap"] < 1600)), s["last_lap"]
    n_viol, _ = env.env.debug_violations()
    assert n_viol == 0

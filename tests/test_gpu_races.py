"""GPU: races (OkRaces).  The race pass after every kind of tick against the port oracle with the pass of
tests/race_oracle.py, bit for bit on every buffer and on hit_car and contact (NaN equal to NaN).  The oracle follows whole
populations, so every race is covered whole.  The cars of each race are teleported into lines by buffer writes every few
ticks (overlapping, inside the lidar's 1.4 px crash band, in range and out of it), so car hits and contact crashes happen;
each test asserts that they did.  Also: the fused actor + tick against its two launches, a CUDA graph replay against eager
calls, the host entry points' refusal while races are on, and the self-check count."""
import numpy as np
import pytest
import torch

import openkitchen_b200 as ok
from openkitchen_b200.dlpack import DeviceBuffer
from tests.laps_oracle import Laps
from tests.race_oracle import CONTACT, SENSE, Races, pack_races
from tests.reset_draws_oracle import DrawnResets
from tests.util import assert_same, make_pair, spread_points

pytestmark = pytest.mark.gpu

RADIUS = 4.0
SEED = 0x7ACE


def race_views(env) -> dict:
    return {k: torch.from_dlpack(DeviceBuffer(env, k, info)) for k, info in env.race_buffers_info().items()}


def assert_races(env, races: Races, ctx):
    env.sync()
    got = {k: v.cpu().numpy() for k, v in race_views(env).items()}
    for k, want in (("hit_car", races.hit_car), ("contact", races.contact)):
        bad = np.argwhere(got[k] != want)
        assert bad.size == 0, f"{ctx}: {k}: {len(bad)} mismatches, first at {tuple(bad[0])}: gpu={got[k][tuple(bad[0])]} oracle={want[tuple(bad[0])]}"


def teleport(env, ora, tid, group, rng, nan=()):
    """the cars of every race lined up (tests/race_oracle.pack_races), the same in both; `nan`: agents given a NaN x"""
    x, y, rot = pack_races(ora.buffer("pos_x"), ora.buffer("pos_y"), ora.buffer("rot"), tid, group, rng)
    x[list(nan)] = np.nan
    for name, v in (("pos_x", x), ("pos_y", y), ("rot", rot)):
        env.write(name, v)
        ora.buffer(name)[:] = v


def no_violations(env):
    n, _ = env.debug_violations()
    assert n == 0, f"{n} out-of-range indices counted"


def exercised(races: Races):
    if races.flags & SENSE:
        assert races.car_hits > 0, "no ray hit a car"
    if races.flags & CONTACT:
        assert races.contact_crashes > 0, "no contact crash"
    else:
        assert races.sense_crashes > 0, "no crash from what the lidar saw"


def run(group=8, n=96, rays=16, flags=SENSE | CONTACT, raycast=ok.RAYCAST_BEAM, names=("Monza", "Spa"), grouped=False,
        ticks=40, every=8, tick="random", draws=0, laps=False, auto_reset=1, nan=(), offset=0.0):
    env, ora, tid = make_pair(list(names), n, rays, grouped=grouped, raycast_mode=raycast, reward_mode=ok.REWARD_CMAES_PROGRESS,
                              auto_reset=auto_reset, sensor_offset=offset)
    fan = ok.ray_fan(rays)
    env.set_reset_draw_flags(SEED, draws)
    drawn = DrawnResets(ora, SEED, draws)
    lap = Laps(ora, drawn) if laps else None
    pts = spread_points(ora, tid)
    env.reset(None, pts)
    (lap.reset if lap else ora.reset)(None, pts)
    if lap:
        env.set_laps(1)
        lap.set(True, 1)
    env.set_races(group, RADIUS, sense=bool(flags & SENSE), contact=bool(flags & CONTACT))
    assert env.races() == {"group": group, "radius": RADIUS, "sense": bool(flags & SENSE), "contact": bool(flags & CONTACT)}
    races = Races(ora, fan, group, RADIUS, flags)
    rng = np.random.default_rng(group * 7 + n)
    for step in range(ticks):
        if step % every == 0:
            teleport(env, ora, tid, group, rng, nan if step == 0 else ())
        if tick == "cast" or step % every == 0 and tick == "mixed":
            env.cast_rays()
            ora.cast_rays()
        else:
            if tick == "steps":
                env.launch_steps_random(step, 1)
            else:
                env.fill_random_actions(step)
                env.launch_step()
            ora.fill_random_actions(step)
            (lap.step if lap else drawn.step)()
        races.apply()
        if step % 4 == 3 or step == ticks - 1:
            assert_same(env, ora, ctx=f"tick {step}")
            assert_races(env, races, f"tick {step}")
    exercised(races)
    no_violations(env)
    return env, ora, races


@pytest.mark.parametrize("kernel", ["staged", "unstaged"])
def test_beam_kernel_shapes(kernel, monkeypatch):
    monkeypatch.setenv("OK_BEAM_KERNEL", kernel)
    env, _, _ = run(tick="mixed")
    assert (env.launch_stats().block_threads == 1024) == (kernel == "staged")


@pytest.mark.parametrize("raycast", [ok.RAYCAST_GRID, ok.RAYCAST_BRUTE])
def test_grid_and_brute_modes(raycast):
    run(raycast=raycast, tick="mixed")


@pytest.mark.parametrize("group,n", [(2, 64), (7, 100), (32, 160), (1024, 1100)])
def test_groups(group, n):
    """a ragged last race at 7 (100 = 14 * 7 + 2) and at 1,024 (1,100 = 1,024 + 76); tracks in two contiguous halves, so
    most races are on one track and one mixes both"""
    run(group=group, n=n, rays=8 if group == 1024 else 16, ticks=24 if group == 1024 else 40, grouped=True)


@pytest.mark.parametrize("flags", [SENSE, CONTACT])
def test_sense_only_and_contact_only(flags):
    _, _, races = run(flags=flags)
    if flags == CONTACT:
        assert np.all(races.hit_car == -1)


def test_races_that_mix_tracks_and_sensor_offset():
    """four tracks interleaved, so every race of 8 mixes them; a sensor offset moves the lidar origin off pos_"""
    run(names=("Monza", "Spa", "Silverstone", "Austin"), offset=3.0)


def test_rays_above_32():
    run(rays=40, n=48, ticks=16)


def test_cast_rays_only_and_origins_inside_bodies():
    """ok_cast_rays with cars teleported so that some lidar origins lie inside the car ahead (t = 0)"""
    _, _, races = run(tick="cast", ticks=16, every=4)
    assert races.inside_hits > 0


def test_nan_poses():
    run(nan=(1, 5, 40), ticks=8)


@pytest.mark.parametrize("draws", [0, 7])
def test_auto_reset_laps_and_steps_random(draws):
    """auto-reset by the stride rule and by drawn resets, lap accounting on, ticks of ok_launch_steps_random"""
    run(draws=draws, laps=True, tick="steps", ticks=48)


def test_step_host_is_refused_while_races_are_on():
    env, ora, tid = make_pair(["Monza"], 32, 8, auto_reset=1)
    thr = np.zeros(32, np.float32)
    obs = np.zeros((32, 8), np.float32)
    env.step_host(thr, thr, obs)
    env.set_races(8, RADIUS)
    with pytest.raises(ok.OkError) as ex:
        env.step_host(thr, thr, obs)
    assert ex.value.code == ok._capi.OK_ERR_STATE
    env.set_races(0)
    env.step_host(thr, thr, obs)
    assert env.races()["group"] == 0


def test_launch_count_is_unchanged_with_races_off():
    env, _, _ = make_pair(["Monza"], 64, 8)
    before = env.launch_stats().kernel_launches
    env.launch_steps_random(0, 5)
    assert env.launch_stats().kernel_launches - before == 5
    env.set_races(8, RADIUS)
    env.launch_steps_random(5, 5)
    assert env.launch_stats().kernel_launches - before == 15


def _batch(n=128, rays=8):
    e = ok.BatchEnv(["Monza", "Spa"], n, rays=rays, reward_mode=ok.REWARD_CONSTANT, auto_reset=1,
                    track_id=(np.arange(n) % 2).astype(np.int32))
    e.set_reset_draws(SEED, point=True, lane=True, heading=True)
    e.set_races(8, RADIUS)
    assert e.race_settings()["group"] == 8 and e.hit_car.shape == (n, rays) and e.contact.shape == (n,)
    return e


def _teleport_batch(envs, seed):
    e0 = envs[0]
    tid = e0.track_id.numpy()
    x, y, rot = pack_races(e0.pos_x.cpu().numpy(), e0.pos_y.cpu().numpy(), e0.rot.cpu().numpy(), tid, 8,
                           np.random.default_rng(seed))
    for e in envs:
        for v, new in ((e.pos_x, x), (e.pos_y, y), (e.rot, rot)):
            v.copy_(torch.from_numpy(new).to(v.device))
    torch.cuda.synchronize()


def _same_envs(a, b, ctx):
    for nm in ok.BUFFERS:
        assert torch.equal(a[nm].view(torch.uint8), b[nm].view(torch.uint8)), (nm, ctx)
    assert torch.equal(a.hit_car, b.hit_car) and torch.equal(a.contact, b.contact), ctx


def test_fused_actor_step_equals_actor_plus_step():
    from openkitchen_b200.rollout import FusedActorRollout

    a, b = _batch(), _batch()
    g = torch.Generator().manual_seed(0)
    l1, l2 = torch.nn.Linear(a.n_rays, 16), torch.nn.Linear(16, 5)
    with torch.no_grad():
        for m in (l1, l2):
            m.weight.copy_(torch.randn(m.weight.shape, generator=g) * 0.5)
            m.bias.copy_(torch.randn(m.bias.shape, generator=g) * 0.1)
    l1, l2 = l1.to(a.device), l2.to(a.device)
    table = torch.tensor([[0.0, 0.0], [80.0, 0.0], [80.0, 4.0], [80.0, -4.0], [40.0, 2.0]])
    ra = FusedActorRollout(a, l1, l2, table, 6, one_launch=True)
    rb = FusedActorRollout(b, l1, l2, table, 6, one_launch=False)
    hits = contacts = 0
    for rnd in range(6):
        _teleport_batch([a, b], rnd)
        ra.run_eager()
        rb.run_eager()
        torch.cuda.synchronize()
        _same_envs(a, b, f"round {rnd}")
        assert torch.equal(ra.actions, rb.actions) and torch.equal(ra.dones, rb.dones)
        hits += int((a.hit_car >= 0).sum())
        contacts += int(a.contact.sum())
    assert hits > 0 and contacts > 0
    no_violations(a.env)


def test_graph_replay_equals_eager_calls():
    a, c = _batch(), _batch()
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(g, stream=side):
            for _ in range(3):
                a.step_random(1)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    a.set_races(0)  # the graph keeps the settings it was captured with
    contacts = hits = 0
    for rnd in range(8):
        _teleport_batch([a, c], 100 + rnd)
        g.replay()
        for t in range(3):
            c.env.launch_steps_random(t, 1, stream=c._stream())
            hits += int((c.hit_car >= 0).sum())
            contacts += int(c.contact.sum())
        torch.cuda.synchronize()
        _same_envs(a, c, f"replay {rnd}")
    assert hits > 0 and contacts > 0

"""GPU: index self-checks.  With the product library this only asserts that the checks are compiled out; run through
tools/checked_build.sh (OK_B200_LIB = a -DOK_CHECKED=1 build) the same workload range-checks every table row, chunk,
segment, ray and agent index in the beam kernels and must count zero violations (the pool's compute-sanitizer is closed)."""
import numpy as np
import pytest
import torch

import openkitchen_b200 as ok
from openkitchen_b200.rollout import FusedActorRollout

pytestmark = pytest.mark.gpu


def test_no_index_leaves_its_array():
    names = ["Spa", "Monza", "Sepang", "Austin", "Oschersleben"]
    for n, offset in ((2560, 0.0), (2304, 4.0), (160, -3.0)):  # staged kernel, with sensor offset, unstaged kernel
        env = ok.Env(device=0, reward_mode=ok.REWARD_CMAES_PROGRESS, auto_reset=1, sensor_offset=offset)
        for nm in names:
            env.add_named_track(nm)
        env.alloc_agents(n, ok.ray_fan(32), (np.arange(n) * len(names) // n).astype(np.int32))
        env.launch_steps_random(0, 60)
        # poses far outside the lane and non-finite ones take the uncovered / grid-walk paths
        x = env.read("pos_x")
        x[::7] += 500.0
        x[3::97] = np.nan
        env.write("pos_x", x)
        env.write("crashed", np.zeros(n, dtype=np.uint8))
        env.launch_steps_random(60, 5)
        count, compiled_in = env.debug_violations()
        assert count == 0, f"{count} out-of-range indices"
        env.close()
    if not compiled_in:
        assert ok.LIB_PATH.endswith("libopenkitchen_b200.so")


def test_no_index_leaves_its_array_in_the_fused_actor_tick():
    """The unstaged beam kernel with the PPO racers' policy step fused in (one launch per tick) has a self-check counter
    of its own: a small population selects that shape."""
    torch.manual_seed(0)
    l1, l2 = torch.nn.Linear(5, 128).cuda(), torch.nn.Linear(128, 3).cuda()
    table = torch.tensor([[60.0, 0.0], [30.0, 5.0], [30.0, -5.0]], device="cuda")
    n = 300
    env = ok.BatchEnv(["Monza", "Zandvoort"], n, rays=np.array([-70, -30, 0, 30, 70], dtype=np.float32),
                      reward_mode=ok.REWARD_CONSTANT, auto_reset=1)
    env.reset(None, torch.from_numpy((np.arange(n) * 53 % 600).astype(np.int32)).cuda())
    env.cast_rays()
    before = env.env.launch_stats().kernel_launches
    FusedActorRollout(env, l1, l2, table, steps=40, sample=True, one_launch=True).run_eager()
    torch.cuda.synchronize()
    assert env.env.launch_stats().kernel_launches - before == 41  # one launch per tick: the fused kernel ran
    count, compiled_in = env.env.debug_violations()
    assert count == 0, f"{count} out-of-range indices"
    env.close()
    if not compiled_in:
        assert ok.LIB_PATH.endswith("libopenkitchen_b200.so")

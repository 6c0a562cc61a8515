"""Evaluation driver (SURVEY §8(f) rank 3): circle_test.enjoy and generate_action_no_sampling against the reference's
semantics (circle_test.py:36-84, model/ppo.py:84-107) with the reference's shipped stage2.pth (large matrices sampled,
tests/golden/checkpoints_sampled.npz)."""
import os
import sys

import numpy as np
import pytest
import torch

from golden_inputs import shipped_checkpoint
from helpers import make_pair

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _policy(n):
    from rl_collision_avoidance_b200.model.net import CNNPolicy
    pol = CNNPolicy(frames=3, action_space=2, max_batch=n)
    pol.load_state_dict({k: torch.from_numpy(v) for k, v in shipped_checkpoint('stage2')[0].items()})
    return pol


def test_generate_action_no_sampling_is_the_clipped_mean(built):
    """model/ppo.py:84-107: mean of the policy, scaled_action = clip(mean, action_bound) - no sampling noise."""
    from rl_collision_avoidance_b200.model.ppo import generate_action_no_sampling
    sc, env, orc = make_pair('circle', num_worlds=1, auto_reset=0, seed=0)
    env.reset_pose()
    pol = _policy(env.N)
    obs = env.get_laser_observation()
    stack = obs[:, None, :].repeat(1, 3, 1).contiguous()
    bound = [[0, -1], [1, 1]]
    mean, scaled = generate_action_no_sampling(env=env, state_list=(stack, env.get_local_goal(), env.get_self_speed()),
                                               policy=pol, action_bound=bound)
    mean2, scaled2 = generate_action_no_sampling(env=env, state_list=(stack, env.get_local_goal(), env.get_self_speed()),
                                                 policy=pol, action_bound=bound)
    assert torch.equal(mean, mean2) and torch.equal(scaled, scaled2)                 # deterministic
    _, ref_mean = pol.forward_values(stack.view(env.N, -1), pol._pack_gs(env.get_local_goal(), env.get_self_speed()))
    assert torch.equal(mean, ref_mean)
    lo, hi = torch.tensor(bound[0], device='cuda'), torch.tensor(bound[1], device='cuda')
    assert torch.equal(scaled, torch.minimum(torch.maximum(mean, lo.float()), hi.float()))
    assert float(mean[:, 0].min()) >= 0.0 and float(mean[:, 0].max()) <= 1.0         # sigmoid head
    assert float(mean[:, 1].abs().max()) <= 1.0                                       # tanh head


def test_enjoy_follows_the_reference_loop(built):
    """50 ticks of circle_test.enjoy on 2 worlds: replayed tick by tick on the CPU oracle with the actions recomputed
    from the oracle's own observations (policy mean on the GPU, terminal robots get v = 0 from the PREVIOUS tick's
    terminate flag, circle_test.py:64-70).  The env state after enjoy must equal the oracle's, bit for bit."""
    sys.path.insert(0, ROOT)
    import circle_test
    sc, env, orc = make_pair('circle', num_worlds=2, auto_reset=0, seed=4)
    pol = _policy(env.N)
    bound = [[0, -1], [1, 1]]
    ever, result, steps_to_end, steps = circle_test.enjoy(env, pol, bound, 50)
    torch.cuda.synchronize()
    # the same loop on the oracle
    orc.reset_world()
    orc.reset_pose()
    N = orc.N
    stack = np.repeat(orc.obs[:, None, :], 3, axis=1).copy()
    terminal = np.zeros(N, bool)
    ever_ref = np.zeros(N, bool)
    for step in range(1, steps + 1):
        gs = torch.from_numpy(orc.gs.copy()).cuda()
        _, mean = pol.forward_values(torch.from_numpy(stack).cuda().view(N, -1), gs)
        a = torch.minimum(torch.maximum(mean, torch.tensor([0.0, -1.0], device='cuda')), torch.tensor([1.0, 1.0], device='cuda'))
        a = a.cpu().numpy().copy()
        a[terminal, 0] = 0.0
        orc.step(a)
        terminal = orc.flags[:, 0] != 0
        ever_ref |= terminal
        stack = np.stack([stack[:, 1], stack[:, 2], orc.obs], 1)
    st = env.state
    for k, ref in (('pose', orc.pose), ('goal', orc.goal), ('acc', orc.acc), ('meta', orc.meta)):
        assert np.array_equal(st[k].cpu().numpy().view(np.uint32), ref.view(np.uint32)), k
    assert np.array_equal(env.obs.cpu().numpy().view(np.uint32), orc.obs.view(np.uint32))
    assert np.array_equal(ever.cpu().numpy(), ever_ref)
    assert steps == 50 or ever_ref.all()
    moved = np.hypot(orc.pose[:, 0] - orc.init_tab[np.arange(N) % 50, 0], orc.pose[:, 1] - orc.init_tab[np.arange(N) % 50, 1])
    assert moved.max() > 1.0                                                          # the trained policy drives off the circle

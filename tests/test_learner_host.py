"""Host-side learner logic vs the reference's golden vectors (no GPU needed)."""
import os

import numpy as np
import torch

GOLD = os.path.join(os.path.dirname(__file__), 'golden', 'learner_golden.npz')


def test_get_filter_index_matches_reference_including_counter_leak():
    from rl_collision_avoidance_b200.model.utils import get_filter_index
    g = np.load(GOLD)
    got = get_filter_index(g['filter_dlist'])
    assert sorted(got) == sorted(g['filter_index'].tolist())
    assert got == g['filter_index'].tolist()          # same order as the reference's loops
    assert get_filter_index(torch.from_numpy(g['filter_dlist'])) == got
    # a column ending in True leaks into the next column's first step (SURVEY App. D.6)
    d = np.zeros((3, 2), bool)
    d[2, 0] = True
    d[0, 1] = True
    assert get_filter_index(d) == [1]


def test_get_group_terminal():
    from rl_collision_avoidance_b200.model.utils import GROUP_REFER, get_group_terminal
    t = np.zeros(44, bool)
    t[0:6] = True                   # group 0 complete
    t[6:9] = True                   # group 1 incomplete
    out = get_group_terminal(t)
    assert out[:6].all() and not out[6:].any()
    assert get_group_terminal(t, index=3) is True and get_group_terminal(t, index=7) is False
    t2 = np.stack([t, np.ones(44, bool)])
    out2 = get_group_terminal(torch.from_numpy(t2))
    assert out2[1].all() and out2[0, :6].all() and not out2[0, 6:].any()
    assert GROUP_REFER == [0, 6, 10, 15, 19, 24, 34, 44]


def test_log_normal_density():
    from rl_collision_avoidance_b200.model.utils import log_normal_density
    x = torch.tensor([[0.7, 0.1]])
    mean = torch.tensor([[0.5, 0.0]])
    ls = torch.tensor([[-1.0, -0.5]])
    got = log_normal_density(x, mean, ls, torch.exp(ls))
    ref = sum(-(xx - m) ** 2 / (2 * np.exp(2 * l)) - 0.5 * np.log(2 * np.pi) - l
              for xx, m, l in ((0.7, 0.5, -1.0), (0.1, 0.0, -0.5)))
    assert abs(got.item() - ref) < 1e-6


def test_golden_file_is_from_the_reference():
    g = np.load(GOLD)
    # SURVEY App. C known answer for generate_train_data
    assert np.allclose(g['gae_small_targets'], [[1.0198, 3.592677], [0.0, 3.788385], [1.099, 1.891]], atol=1e-6)
    assert np.allclose(g['gae_small_advs'], [[0.5198, 3.092677], [-0.4, 3.188385], [0.799, 1.691]], atol=1e-6)
    assert g['ppo_losses'].shape == (3, 3)


def test_stage2_golden_filter_is_our_filter():
    """The rows the reference's ppo_update_stage2 golden deleted are get_filter_index of the same done flags."""
    import sys
    sys.path.insert(0, os.path.dirname(__file__))
    from golden_inputs import stage2_rollout
    from rl_collision_avoidance_b200.model.utils import get_filter_index
    g = np.load(GOLD)
    assert [int(i) for i in get_filter_index(stage2_rollout()['dones'])] == g['ppo2_filter_index'].tolist()
    n_kept = 48 - len(g['ppo2_filter_index'])
    assert g['ppo2_perms'].shape == (2, n_kept) and n_kept % int(g['ppo2_batch_size']) != 0


def test_reference_checkpoint_fixtures_have_the_23_tensors():
    """tests/golden/checkpoints_sampled.npz holds the reference's shipped policy/*.pth (data fixtures, the large
    matrices sampled): same keys, key order and shapes as our flat parameter layout (SURVEY App. C)."""
    sys_path = os.path.dirname(__file__)
    import sys
    sys.path.insert(0, sys_path)
    from golden_inputs import SHAPES, shipped_checkpoint
    for name in ('stage1_1', 'stage1_2', 'stage2'):
        sd, _ = shipped_checkpoint(name)
        assert [(k, tuple(v.shape)) for k, v in sd.items()] == [(k, tuple(s)) for k, s in SHAPES]
        assert all(v.dtype == np.float32 for v in sd.values())


def test_transform_buffer_matches_reference_golden():
    """model/ppo.py:22-54: the rollout buffer (per step: states of every robot, action, reward, done, logprob, value)
    stacked into eight (T, N, ...) arrays.  The reference's own function ran on a seeded buffer
    (tools/make_golden_buffer.py -> tests/golden/buffer_golden.npz); ours takes the per-step BATCHED form of the same
    data and must return the same eight arrays in the same order."""
    import os
    import torch
    from rl_collision_avoidance_b200.model.ppo import transform_buffer
    g = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'buffer_golden.npz'))
    T = g['in_obs'].shape[0]
    buff = []
    for t in range(T):
        state = (torch.from_numpy(g['in_obs'][t]), torch.from_numpy(g['in_goal'][t]), torch.from_numpy(g['in_speed'][t]))
        buff.append((state, torch.from_numpy(g['in_a'][t]), torch.from_numpy(g['in_r'][t]), torch.from_numpy(g['in_d'][t]),
                     torch.from_numpy(g['in_l'][t]), torch.from_numpy(g['in_v'][t])))
    got = transform_buffer(buff)
    assert len(got) == 8
    for name, arr in zip(('s', 'goal', 'speed', 'a', 'r', 'd', 'l', 'v'), got):
        ref = g['out_' + name]
        assert tuple(arr.shape) == ref.shape, name
        assert np.array_equal(arr.numpy(), ref), name

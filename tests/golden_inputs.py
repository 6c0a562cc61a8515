"""Deterministic synthetic weights / batches shared by tools/make_golden.py (reference side) and the GPU tests
(our side).  Everything is derived from numpy RandomState streams, which are stable across numpy versions."""
import os

import numpy as np

SHAPES = [
    ('logstd', (2,)),
    ('act_fea_cv1.weight', (32, 3, 5)), ('act_fea_cv1.bias', (32,)),
    ('act_fea_cv2.weight', (32, 32, 3)), ('act_fea_cv2.bias', (32,)),
    ('act_fc1.weight', (256, 4096)), ('act_fc1.bias', (256,)),
    ('act_fc2.weight', (128, 260)), ('act_fc2.bias', (128,)),
    ('actor1.weight', (1, 128)), ('actor1.bias', (1,)),
    ('actor2.weight', (1, 128)), ('actor2.bias', (1,)),
    ('crt_fea_cv1.weight', (32, 3, 5)), ('crt_fea_cv1.bias', (32,)),
    ('crt_fea_cv2.weight', (32, 32, 3)), ('crt_fea_cv2.bias', (32,)),
    ('crt_fc1.weight', (256, 4096)), ('crt_fc1.bias', (256,)),
    ('crt_fc2.weight', (128, 260)), ('crt_fc2.bias', (128,)),
    ('critic.weight', (1, 128)), ('critic.bias', (1,)),
]


def shipped_checkpoint(name):
    """The reference's shipped policy/<name>.pth as shrunk by tools/make_golden_checkpoints.py: (state_dict of numpy
    arrays with the shipped keys, order, shapes and dtypes; the reference CNNPolicy's App. C probes on those weights)."""
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'checkpoints_sampled.npz'))
    sd = {k.split(':', 1)[1]: z[k] for k in z.files if k.startswith(name + ':') and k != name + ':probe'}
    return sd, z[name + ':probe']


def synthetic_state_dict(seed=1234):
    rs = np.random.RandomState(seed)
    sd = {}
    for name, shape in SHAPES:
        if name == 'logstd':
            sd[name] = np.array([-0.3, -0.7], np.float32)
            continue
        fan_in = int(np.prod(shape[1:])) if len(shape) > 1 else int(np.prod(dict(SHAPES)[name.replace('bias', 'weight')][1:]))
        sd[name] = (rs.uniform(-1, 1, size=shape) / np.sqrt(fan_in) * 1.7).astype(np.float32)
    return sd


def synthetic_batch(nb, seed=99):
    rs = np.random.RandomState(seed)
    base = rs.uniform(-0.5, 0.5, size=(nb, 1, 512))
    obs = np.clip(base + 0.05 * rs.standard_normal((nb, 3, 512)), -0.5, 0.5).astype(np.float32)
    goal = rs.uniform(-8, 8, size=(nb, 2)).astype(np.float32)
    speed = np.stack([rs.uniform(0, 1, nb), rs.uniform(-1, 1, nb)], 1).astype(np.float32)
    action = np.stack([rs.uniform(-0.2, 1.2, nb), rs.uniform(-1.2, 1.2, nb)], 1).astype(np.float32)
    return obs, goal, speed, action


def synthetic_rollout(T, N, seed=5, with_obs=False):
    rs = np.random.RandomState(seed)
    out = {
        'rewards': rs.uniform(-1, 1, size=(T, N)).astype(np.float32),
        'values': rs.uniform(-2, 2, size=(T, N)).astype(np.float32),
        'last_value': rs.uniform(-2, 2, size=(N,)).astype(np.float32),
        'dones': (rs.rand(T, N) < 0.2),
    }
    if with_obs:
        obs, goal, speed, action = synthetic_batch(T * N, seed=seed + 1)
        out['obs'] = obs.reshape(T, N, 3, 512)
        out['goal'] = goal.reshape(T, N, 2)
        out['speed'] = speed.reshape(T, N, 2)
        out['action'] = action.reshape(T, N, 2)
        out['logprob'] = rs.uniform(-1.5, 0.5, size=(T, N, 1)).astype(np.float32)
    return out


def stage2_rollout(T=6, N=8):
    """Rollout for the ppo_update_stage2 golden: done flags dense enough (45 %) that get_filter_index finds runs of
    consecutive terminal steps (the rows stage 2 deletes, model/utils.py:65-78)."""
    roll = synthetic_rollout(T=T, N=N, seed=11, with_obs=True)
    roll['dones'] = np.random.RandomState(21).rand(T, N) < 0.45
    return roll

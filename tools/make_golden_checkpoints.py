"""Shrink the reference's shipped checkpoints (policy/*.pth, 8.7 MB each) into one test fixture,
tests/golden/checkpoints_sampled.npz, and record what the reference's own CNNPolicy computes on it.

    python tools/make_golden_checkpoints.py <reference checkout>

Every tensor of up to 4096 entries is kept as shipped (logstd, conv towers, biases, heads).  Of the larger weight
matrices (act/crt_fc1, act/crt_fc2) a seeded 1/256 sample of the entries is kept, scaled by 16 so that the
pre-activations keep their magnitude, and the rest is zero; zeros compress, so the three checkpoints fit in ~0.3 MB.
The keys are written in the order of the shipped state_dict.  `<name>:probe` holds the SURVEY App. C probes (value
and mean for a free and a ramp observation, log-prob and entropy) through the reference's own model/net.py.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEEP = 1.0 / 256
NAMES = ('stage1_1', 'stage1_2', 'stage2')


def shrink(sd, seed):
    rs = np.random.RandomState(seed)
    out = {}
    for k, v in sd.items():
        a = v.numpy().astype(np.float32)
        if a.size > 4096:
            a = np.where(rs.rand(*a.shape) < KEEP, a / np.float32(np.sqrt(KEEP)), np.float32(0)).astype(np.float32)
        out[k] = a
    return out


def main(ref):
    torch.set_num_threads(4)
    cwd = os.getcwd()
    sys.path.insert(0, ref)
    from model.net import CNNPolicy
    os.chdir(cwd)
    free_obs = torch.full((1, 3, 512), 0.5)
    ramp_obs = (torch.arange(512, dtype=torch.float32) / 511 - 0.5).view(1, 1, 512).repeat(1, 3, 1)
    out = {}
    for i, name in enumerate(NAMES):
        sd = shrink(torch.load(os.path.join(ref, 'policy', name + '.pth'), map_location='cpu'), seed=i)
        pol = CNNPolicy(frames=3, action_space=2)
        pol.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
        with torch.no_grad():
            v_f, _, _, m_f = pol(free_obs, torch.tensor([[5.0, 0.0]]), torch.tensor([[0.0, 0.0]]))
            v_r, _, _, m_r = pol(ramp_obs, torch.tensor([[3.0, -1.0]]), torch.tensor([[0.5, 0.2]]))
            _, lp, ent = pol.evaluate_actions(free_obs, torch.tensor([[5.0, 0.0]]), torch.tensor([[0.0, 0.0]]),
                                              torch.tensor([[0.7, 0.1]]))
        for k, v in sd.items():
            out[f'{name}:{k}'] = v
        out[f'{name}:probe'] = np.array([v_f.item(), m_f[0, 0].item(), m_f[0, 1].item(), v_r.item(), m_r[0, 0].item(),
                                         m_r[0, 1].item(), lp.item(), ent.item()], np.float64)
        print(name, out[f'{name}:probe'])
    path = os.path.join(ROOT, 'tests', 'golden', 'checkpoints_sampled.npz')
    np.savez_compressed(path, **out)
    print('wrote', path, os.path.getsize(path), 'bytes')


if __name__ == '__main__':
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(sys.argv[1])

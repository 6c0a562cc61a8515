"""Generate golden vectors for the learning half from the reference's OWN code.

Run HERE (where /root/reference exists): python tools/make_golden.py
Imports /root/reference/model/{net,ppo,utils}.py unmodified (read-only), with `.cuda()` neutralised because
this container has no GPU, and writes tests/golden/learner_golden.npz.  The GPU tests rebuild the same
synthetic weights/inputs from the same numpy RandomState seeds and compare our kernels against these numbers.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get('RLCA_REFERENCE', '/root/reference')
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

from golden_inputs import stage2_rollout, synthetic_state_dict, synthetic_batch, synthetic_rollout  # noqa: E402


def main():
    torch.set_num_threads(4)
    torch.Tensor.cuda = lambda self, *a, **k: self          # no GPU here
    torch.nn.Module.cuda = lambda self, *a, **k: self
    cwd = os.getcwd()
    os.chdir('/tmp')                                         # model/ppo.py creates ./log/<host>/ at import
    sys.path.insert(0, REF)
    import functools
    import builtins
    builtins.reduce = functools.reduce                       # py2 builtin used by model/utils.py:85
    from model.net import CNNPolicy
    from model import ppo as ref_ppo
    from model import utils as ref_utils
    os.chdir(cwd)
    out = {}

    # ---- policy forward / evaluate_actions on synthetic weights
    sd = synthetic_state_dict()
    pol = CNNPolicy(frames=3, action_space=2)
    pol.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    obs, goal, speed, action = synthetic_batch(16)
    with torch.no_grad():
        v, logp, ent = pol.evaluate_actions(torch.from_numpy(obs), torch.from_numpy(goal), torch.from_numpy(speed),
                                            torch.from_numpy(action))
        _, _, _, mean = pol(torch.from_numpy(obs), torch.from_numpy(goal), torch.from_numpy(speed))
    out['fwd_value'] = v.numpy()
    out['fwd_mean'] = mean.numpy()
    out['fwd_logprob'] = logp.numpy()
    out['fwd_entropy'] = np.float64(ent.item())

    # ---- GAE (generate_train_data, model/ppo.py:122-139): SURVEY App. C known answer + a random case
    r = np.array([[1, 0], [0, 2], [1, 1]], np.float64)
    vals = np.array([[.5, .5], [.4, .6], [.3, .2]], np.float64)
    d = np.array([[0, 0], [1, 0], [0, 0]], np.float64)
    t, a = ref_ppo.generate_train_data(r, 0.99, vals, np.array([.1, .9]), d, 0.95)
    out['gae_small_targets'], out['gae_small_advs'] = t, a
    roll = synthetic_rollout(T=24, N=7)
    t, a = ref_ppo.generate_train_data(roll['rewards'].astype(np.float64), 0.99, roll['values'].astype(np.float64),
                                       roll['last_value'].astype(np.float64), roll['dones'].astype(np.float64), 0.95)
    out['gae_targets'], out['gae_advs'] = t, a

    # ---- get_filter_index (model/utils.py:65-78) incl. the cross-column counter leak
    rs = np.random.RandomState(7)
    dl = rs.rand(12, 6) < 0.45
    dl[-1, 2] = True
    dl[0, 3] = True
    out['filter_dlist'] = dl
    out['filter_index'] = np.asarray(ref_utils.get_filter_index(dl), np.int64)

    # ---- ppo_update_stage1 (model/ppo.py:143-194): one minibatch == the whole set, so sampling order is irrelevant
    T, N = 4, 8
    roll = synthetic_rollout(T=T, N=N, with_obs=True)
    pol = CNNPolicy(frames=3, action_space=2)
    pol.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    opt = torch.optim.Adam(pol.parameters(), lr=5e-5)
    tg, adv = ref_ppo.generate_train_data(roll['rewards'].astype(np.float64), 0.99, roll['values'].astype(np.float64),
                                          roll['last_value'].astype(np.float64), roll['dones'].astype(np.float64), 0.95)
    memory = (roll['obs'].astype(np.float64), roll['goal'].astype(np.float64), roll['speed'].astype(np.float64),
              roll['action'], roll['logprob'], tg, roll['values'], roll['rewards'], adv)
    rows = []

    class Cap:
        def info(self, msg):
            rows.append([float(x) for x in msg.split(',')])
    ref_ppo.logger_ppo = Cap()
    ref_ppo.ppo_update_stage1(policy=pol, optimizer=opt, batch_size=T * N, memory=memory, epoch=3, coeff_entropy=5e-4,
                              clip_value=0.1, num_step=T, num_env=N, frames=3, obs_size=512, act_size=2)
    out['ppo_losses'] = np.asarray(rows, np.float64)
    after = pol.state_dict()
    out['ppo_logstd_after'] = after['logstd'].numpy()
    for k in ('act_fea_cv1.weight', 'act_fea_cv2.bias', 'act_fc1.bias', 'act_fc2.weight', 'actor1.weight', 'actor2.bias',
              'crt_fea_cv1.bias', 'crt_fea_cv2.weight', 'crt_fc2.bias', 'critic.weight', 'critic.bias'):
        out['ppo_after_' + k] = after[k].numpy()
    out['ppo_after_act_fc1.weight_rows'] = after['act_fc1.weight'].numpy()[::37, ::301]
    out['ppo_after_crt_fc1.weight_rows'] = after['crt_fc1.weight'].numpy()[::41, ::307]

    # ---- gradient of the first step's loss (for the backward kernels)
    pol = CNNPolicy(frames=3, action_space=2)
    pol.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    advn = (adv - adv.mean()) / adv.std()
    ft = lambda x: torch.from_numpy(np.asarray(x)).float()
    nv, nl, ent = pol.evaluate_actions(ft(roll['obs'].reshape(T * N, 3, 512)), ft(roll['goal'].reshape(T * N, 2)),
                                       ft(roll['speed'].reshape(T * N, 2)), ft(roll['action'].reshape(T * N, 2)))
    ratio = torch.exp(nl - ft(roll['logprob'].reshape(T * N, 1)))
    A = ft(advn.reshape(T * N, 1))
    pl = -torch.min(ratio * A, torch.clamp(ratio, 0.9, 1.1) * A).mean()
    vl = torch.nn.functional.mse_loss(nv, ft(tg.reshape(T * N, 1)))
    loss = pl + 20 * vl - 5e-4 * ent
    loss.backward()
    g = {k: p.grad.numpy() for k, p in pol.named_parameters()}
    out['grad_logstd'] = g['logstd']
    for k in ('act_fea_cv1.weight', 'act_fea_cv1.bias', 'act_fea_cv2.weight', 'act_fea_cv2.bias', 'act_fc1.bias',
              'act_fc2.weight', 'act_fc2.bias', 'actor1.weight', 'actor1.bias', 'actor2.weight', 'actor2.bias',
              'crt_fea_cv1.weight', 'crt_fea_cv1.bias', 'crt_fea_cv2.weight', 'crt_fea_cv2.bias', 'crt_fc1.bias',
              'crt_fc2.weight', 'crt_fc2.bias', 'critic.weight', 'critic.bias'):
        out['grad_' + k] = g[k]
    out['grad_act_fc1.weight_rows'] = g['act_fc1.weight'][::37, ::301]
    out['grad_crt_fc1.weight_rows'] = g['crt_fc1.weight'][::41, ::307]
    out['loss0'] = np.array([pl.item(), vl.item(), ent.item()])

    # ---- ppo_update_stage2 (model/ppo.py:197-259): rows in filter_index deleted after the normalisation over ALL rows
    # (:200 before :212-218), BatchSampler(drop_last=True) (:221-223) so the ragged tail of every epoch is skipped.
    # The minibatch membership depends on torch.randperm inside SubsetRandomSampler; the permutations the reference drew
    # are recorded so that our side replays exactly the same minibatches.
    T2, N2 = 6, 8
    roll2 = stage2_rollout(T2, N2)
    pol = CNNPolicy(frames=3, action_space=2)
    pol.load_state_dict({k: torch.from_numpy(v) for k, v in sd.items()})
    opt = torch.optim.Adam(pol.parameters(), lr=5e-5)
    tg2, adv2 = ref_ppo.generate_train_data(roll2['rewards'].astype(np.float64), 0.99, roll2['values'].astype(np.float64),
                                            roll2['last_value'].astype(np.float64), roll2['dones'].astype(np.float64), 0.95)
    filt = ref_utils.get_filter_index(roll2['dones'])
    assert len(filt) >= 3, filt                               # the filter must be non-trivial
    memory2 = (roll2['obs'].astype(np.float64), roll2['goal'].astype(np.float64), roll2['speed'].astype(np.float64),
               roll2['action'], roll2['logprob'], tg2, roll2['values'], roll2['rewards'], adv2)
    perms = []
    real_randperm = torch.randperm

    def rec_randperm(n, *a, **k):
        p = real_randperm(n, *a, **k)
        perms.append(p.numpy().copy())
        return p
    torch.randperm = rec_randperm
    torch.manual_seed(2024)
    rows = []
    bs2 = 16
    try:
        ref_ppo.ppo_update_stage2(policy=pol, optimizer=opt, batch_size=bs2, memory=memory2, filter_index=filt, epoch=2,
                                  coeff_entropy=5e-4, clip_value=0.1, num_step=T2, num_env=N2, frames=3, obs_size=512,
                                  act_size=2)
    finally:
        torch.randperm = real_randperm
    n_kept = T2 * N2 - len(filt)
    assert len(perms) == 2 and all(len(p) == n_kept for p in perms), (len(perms), n_kept)
    assert n_kept % bs2 != 0 and len(rows) == 2 * (n_kept // bs2), (n_kept, len(rows))     # ragged tail dropped
    out['ppo2_filter_index'] = np.asarray(filt, np.int64)
    out['ppo2_perms'] = np.stack(perms).astype(np.int64)
    out['ppo2_batch_size'] = np.int64(bs2)
    out['ppo2_losses'] = np.asarray(rows, np.float64)
    after = pol.state_dict()
    out['ppo2_logstd_after'] = after['logstd'].numpy()
    for k in ('act_fea_cv1.weight', 'act_fea_cv2.bias', 'act_fc1.bias', 'act_fc2.weight', 'actor1.weight', 'actor2.bias',
              'crt_fea_cv1.bias', 'crt_fea_cv2.weight', 'crt_fc2.bias', 'critic.weight', 'critic.bias'):
        out['ppo2_after_' + k] = after[k].numpy()
    out['ppo2_after_act_fc1.weight_rows'] = after['act_fc1.weight'].numpy()[::37, ::301]
    out['ppo2_after_crt_fc1.weight_rows'] = after['crt_fc1.weight'].numpy()[::41, ::307]

    path = os.path.join(ROOT, 'tests', 'golden', 'learner_golden.npz')
    np.savez_compressed(path, **out)
    print('wrote', path, {k: np.asarray(v).shape for k, v in out.items() if k.startswith(('fwd', 'ppo_losses', 'loss0'))})
    print('ppo losses', out['ppo_losses'])


if __name__ == '__main__':
    main()

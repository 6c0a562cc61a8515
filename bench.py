#!/usr/bin/env python
"""bench.py — agent-steps/s of the fused simulator tick at 4096 robots x 512 beams.

Contract (driver): `python bench.py --gpus N --steps K --warmup W` (under torchrun for N>1)
prints ONE JSON line on rank 0.  A "step" is one fused tick (integrate + collide + 512-beam
lidar + reward/done + obs) over the per-GPU agent batch: 171 stage-1 worlds x 24 robots =
4104 agents (BASELINE.md §5).  Scaling is weak: every GPU gets its own 171 worlds, no
data-path collective (worlds are independent; SURVEY.md §8(e)).

  value        whole-job agent-steps/s, inputs resident in HBM, CUDA-event timed, max over ranks; the ticks are
               replayed from a CUDA graph (the launch-bound inner loop of a rollout), two kernels per tick
  e2e          same metric through the host-buffer C-ABI call rlca_env_step_host (pinned host buffers in and out,
               PCIe traffic and a stream sync inside every call) — the reference-facing call
  roofline     algorithmic bytes (4*B+96 per agent-step, SURVEY.md §8(d)) / measured per-tick time vs the measured
               HBM copy peak (MEASURED_PEAKS.json, else the 6650 GB/s fallback); traffic = DRAM bytes per launch
               from the committed ncu capture of >= 130 consecutive ring launches (profiles/)
  cpu_baseline the CPU oracle (port of the reference semantics) on the host cores, bounded sample
  sections     (N = 1, outside the timed region, each with its own CPU-oracle figure) the other BASELINE configs:
               stage-2 tick, circle tick, raycast sweep, full PPO training, and the reference learner (stock PyTorch
               fp32) beside ours;  learner_dp (N > 1): the data-parallel minibatch step and its all-reduce share

`--impl reference` times the reference's CPU path.  The literal Stage+ROS+mpi4py stack cannot run here
(BASELINE.md §4), so this is the oracle port with all host threads; it builds and loads the oracle only.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORLDS_PER_GPU = 171
ROBOTS = 24
BEAMS = 512
METRIC = 'agent-steps/s @4096 robots x 512 beams (fused env tick)'
# the workload both arms run (identical string in both JSON lines)
WORKLOAD = (f'stage1 rink arena (100x100 cells @0.2 m), {WORLDS_PER_GPU} worlds x {ROBOTS} robots = '
            f'{WORLDS_PER_GPU * ROBOTS} agents per GPU, {BEAMS} beams, fov pi, range 6 m, dt 0.1 s, '
            'v~U[0,1] w~U[-1,1], auto-reset on done, seed 0')


def alg_bytes(beams):           # SURVEY.md §8(d): the figure builder and judge share
    return 4 * beams + 96


def random_actions(rng, n):
    import numpy as np
    return np.stack([rng.uniform(0.0, 1.0, n), rng.uniform(-1.0, 1.0, n)], 1).astype(np.float32)


def measured_peak():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        try:
            with open(p) as f:
                return float(json.load(f)['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
        except Exception:
            pass
    return 6650.0, 'fallback (B200_PROFILING.md 6.65 TB/s)'


class ClockSampler:
    """Samples SM clocks / throttle reasons with nvidia-smi during the timed region."""
    Q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index=0):
        self.rows = []
        self.proc = None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), f'--query-gpu={self.Q}',
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            parts = [x.strip() for x in r.split(',')]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                mx = float(parts[1])
            except ValueError:
                continue
            for n, v in zip(names, parts[2:6]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        sm.sort()
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': mx, 'reasons': sorted(reasons),
                'samples': len(sm)}


def _cpu_quota():
    """CPUs the cgroup lets this process use (cpu.max), or None."""
    try:
        with open('/sys/fs/cgroup/cpu.max') as f:
            q, per = f.read().split()
        if q != 'max':
            return max(1, int(float(q) / float(per) + 0.5))
    except Exception:
        pass
    return None


# ------------------------------------------------------------------------------------------------ CPU oracle legs
def make_oracle(scenario, num_worlds, beams=BEAMS, auto_reset=True, seed=0, raw_beams=None):
    """The CPU oracle for a scenario (test infrastructure, used here only as the timed CPU baseline)."""
    from oracle.oracle import OracleWorld, OrcConfig
    from rl_collision_avoidance_b200.scenarios import fill_config, make_scenario
    sc = make_scenario(scenario)
    cfg = fill_config(OrcConfig(), sc, num_worlds=num_worlds, beams=beams, raw_beams=raw_beams, auto_reset=auto_reset,
                      seed=seed)
    return OracleWorld(cfg, sc.map.cells, sc.init_tab, sc.goal_tab)


def pick_threads(step_fn, budget_s, threads=None):
    """Fastest sustained OpenMP thread count for `step_fn` (one unit of CPU work).  torchrun exports
    OMP_NUM_THREADS=1 and a cgroup CPU quota can make "all logical CPUs" ~10x slower than fewer threads, but only
    once the quota's burst allowance is gone - so every candidate count runs for a sustained slice."""
    from oracle import oracle as orc_mod
    ncpu = len(os.sched_getaffinity(0))
    quota = _cpu_quota()
    if threads:
        cands = [threads]
    else:
        cands = {max(1, ncpu), max(1, ncpu // 2), max(1, ncpu // 4), min(ncpu, 32), min(ncpu, 16)}
        if quota:
            cands |= {min(ncpu, quota), min(ncpu, max(1, quota // 2))}
        cands = sorted(cands, reverse=True)
    slice_s = max(0.5, min(2.5, budget_s / len(cands)))
    probe = []
    for c in cands:
        orc_mod.set_threads(c)
        step_fn(0)
        n, t0 = 0, time.perf_counter()
        while n < 3 or time.perf_counter() - t0 < slice_s:
            step_fn(n)
            n += 1
        probe.append(((time.perf_counter() - t0) / n, c))
    probe.sort()
    return probe, quota


def run_cpu(steps, warmup, budget_s, threads=None):
    """Time the oracle port on the host cores on the headline workload.
    Returns (agent_steps_per_s, cores, sample_desc, ms_per_tick)."""
    import numpy as np
    from oracle import oracle as orc_mod
    orc = make_oracle('stage1', WORLDS_PER_GPU)
    orc.reset_world()
    orc.reset_pose()
    rng = np.random.default_rng(0)
    acts = [random_actions(rng, orc.N) for _ in range(8)]
    probe, quota = pick_threads(lambda i: orc.step(acts[i % 8]), 0.3 * budget_s, threads)
    best = None
    for t_tick, cores in probe[:2]:
        orc_mod.set_threads(cores)
        worlds = WORLDS_PER_GPU
        total = (steps + warmup) * t_tick
        share = 0.35 * budget_s
        o = orc
        if total > share:
            worlds = min(WORLDS_PER_GPU, max(cores, int(WORLDS_PER_GPU * share / total)))
            o = make_oracle('stage1', worlds)
            o.reset_world()
            o.reset_pose()
        a = [x[:o.N] for x in acts]
        for i in range(warmup):
            o.step(a[i % len(a)])
        t0 = time.perf_counter()
        for i in range(steps):
            o.step(a[i % len(a)])
        dt = time.perf_counter() - t0
        val = o.N * steps / dt
        sample = f'{worlds} of {WORLDS_PER_GPU} stage-1 worlds x {ROBOTS} robots x {BEAMS} beams, {steps} ticks, ' \
                 f'OpenMP over worlds, {cores} threads (best sustained of {sorted(c for _, c in probe)} threads' \
                 f'{", cgroup quota %d CPUs" % quota if quota else ""})'
        if best is None or val > best[0]:
            best = (val, cores, sample, dt / steps * 1e3)
        if val > 0.6 * WORLDS_PER_GPU * ROBOTS / probe[0][0]:      # the sample reproduced the probe: done
            break
    return best


def dump_outputs(out_dir, arrays):
    """Writes each device tensor of `arrays` as out_dir/<name>.npy in float32 (flag bytes are exact in float32)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), t.cpu().numpy().astype(np.float32))


def cpu_sample(fn, units_per_call, cores, seconds=2.5, min_calls=2):
    """units/s of `fn` on the oracle with `cores` threads, for about `seconds` of CPU work."""
    from oracle import oracle as orc_mod
    orc_mod.set_threads(cores)
    fn(0)
    n, t0 = 0, time.perf_counter()
    while n < min_calls or time.perf_counter() - t0 < seconds:
        fn(n + 1)
        n += 1
    return units_per_call * n / (time.perf_counter() - t0), n


# ------------------------------------------------------------------------------------------------ GPU helpers
def gpu_time(torch, dev, fn, n, warm=3):
    """ms per call of fn (CUDA events on the current stream, after warm-up)."""
    for i in range(warm):
        fn(i)
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n):
        fn(i)
    e1.record()
    torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1) / n


def time_learner(dev, n_agents):
    """Side measurement (outside the timed env region, CUDA events): the policy forward at the rollout batch and one
    PPO minibatch step (forward, loss, backward, Adam) at the reference's batch size 1024 (ppo_stage1.py:28)."""
    import torch
    from rl_collision_avoidance_b200 import _lib
    from rl_collision_avoidance_b200.model.net import Adam, CNNPolicy, _ptr
    pol = CNNPolicy(device=str(dev), max_batch=max(n_agents, 1024), seed=0)
    opt = Adam(pol.parameters(), lr=5e-5)
    lib = pol.lib
    out = {'tensor_cores': 'tcgen05 3xTF32: conv tower forward/backward + fc1 forward/dW/dX'}
    for nb, key in ((n_agents, 'policy_forward_us'), (1024, 'ppo_minibatch_step_us')):
        obs = torch.rand(nb, 1536, device=dev) - 0.5
        gs = torch.rand(nb, 4, device=dev)
        v, mean = torch.empty(nb, device=dev), torch.empty(nb, 2, device=dev)
        act, lp = torch.rand(nb, 2, device=dev), torch.rand(nb, device=dev) - 1
        adv, tgt, losses = torch.randn(nb, device=dev), torch.randn(nb, device=dev), torch.zeros(3, device=dev)
        ws, st = pol._workspace(nb), pol._stream()

        def fwd(_=0):
            _lib.check(lib.rlca_policy_forward(ws, _ptr(pol.flat), _ptr(obs), _ptr(gs), nb, _ptr(v), _ptr(mean), st))

        def step(_=0):
            fwd()
            _lib.check(lib.rlca_ppo_loss_fwd_bwd(ws, _ptr(pol.flat), _ptr(v), _ptr(mean), _ptr(act), _ptr(lp), _ptr(adv),
                                                 _ptr(tgt), nb, 0.1, 5e-4, 20.0, _ptr(losses), st))
            _lib.check(lib.rlca_policy_backward(ws, _ptr(pol.flat), _ptr(obs), _ptr(gs), nb, _ptr(pol.grad), st))
            opt.step()

        out[key] = {'batch': nb, 'us': gpu_time(torch, dev, fwd if key == 'policy_forward_us' else step, 10) * 1e3}
    return out


def time_learner_reference(dev, n_agents):
    """The reference's learner through stock PyTorch on the same GPU (BASELINE.md §4.2): CNNPolicy (the architecture of
    /root/reference/model/net.py:16-80 as a plain nn.Module, fp32, TF32 off) forward at the rollout batch, and one
    minibatch step of /root/reference/model/ppo.py:172-188 (evaluate, clipped surrogate + 20 x value - entropy,
    zero_grad, backward, torch.optim.Adam step) at batch 1024."""
    import math
    import torch
    import torch.nn as nn
    import torch.nn.functional as F
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False

    class Ref(nn.Module):
        def __init__(self):
            super().__init__()
            self.logstd = nn.Parameter(torch.zeros(2))
            for p in ('act', 'crt'):
                setattr(self, p + '_fea_cv1', nn.Conv1d(3, 32, 5, 2, 1))
                setattr(self, p + '_fea_cv2', nn.Conv1d(32, 32, 3, 2, 1))
                setattr(self, p + '_fc1', nn.Linear(4096, 256))
                setattr(self, p + '_fc2', nn.Linear(260, 128))
            self.actor1, self.actor2, self.critic = nn.Linear(128, 1), nn.Linear(128, 1), nn.Linear(128, 1)

        def tower(self, p, x, goal, speed):
            h = F.relu(getattr(self, p + '_fea_cv1')(x))
            h = F.relu(getattr(self, p + '_fea_cv2')(h))
            h = F.relu(getattr(self, p + '_fc1')(h.flatten(1)))
            return F.relu(getattr(self, p + '_fc2')(torch.cat((h, goal, speed), -1)))

        def forward(self, x, goal, speed):
            a = self.tower('act', x, goal, speed)
            mean = torch.cat((torch.sigmoid(self.actor1(a)), torch.tanh(self.actor2(a))), -1)
            return self.critic(self.tower('crt', x, goal, speed)), mean

    pol = Ref().to(dev)
    opt = torch.optim.Adam(pol.parameters(), lr=5e-5)
    out = {'impl': 'stock PyTorch eager (cuDNN conv1d + cuBLAS), fp32, allow_tf32 = False', 'torch': torch.__version__}
    nb = n_agents
    x, goal, speed = torch.rand(nb, 3, 512, device=dev) - 0.5, torch.rand(nb, 2, device=dev), torch.rand(nb, 2, device=dev)

    def fwd(_=0):
        with torch.no_grad():
            v, mean = pol(x, goal, speed)
            std = torch.exp(pol.logstd).expand_as(mean)
            a = torch.normal(mean, std)
            return (-(a - mean) ** 2 / (2 * std ** 2) - 0.5 * math.log(2 * math.pi) - pol.logstd).sum(-1)
    out['policy_forward_us'] = {'batch': nb, 'us': gpu_time(torch, dev, fwd, 10) * 1e3}
    nb = 1024
    x, goal, speed = torch.rand(nb, 3, 512, device=dev) - 0.5, torch.rand(nb, 2, device=dev), torch.rand(nb, 2, device=dev)
    act, old_lp = torch.rand(nb, 2, device=dev), torch.rand(nb, 1, device=dev) - 1
    adv, tgt = torch.randn(nb, 1, device=dev), torch.randn(nb, 1, device=dev)

    def step(_=0):
        v, mean = pol(x, goal, speed)
        var = torch.exp(2 * pol.logstd)
        lp = (-(act - mean) ** 2 / (2 * var) - 0.5 * math.log(2 * math.pi) - pol.logstd).sum(-1, keepdim=True)
        ent = (0.5 + 0.5 * math.log(2 * math.pi) + pol.logstd).sum()
        ratio = torch.exp(lp - old_lp)
        pl = -torch.min(ratio * adv, torch.clamp(ratio, 0.9, 1.1) * adv).mean()
        loss = pl + 20 * F.mse_loss(v, tgt) - 5e-4 * ent
        opt.zero_grad()
        loss.backward()
        opt.step()
    out['ppo_minibatch_step_us'] = {'batch': nb, 'us': gpu_time(torch, dev, step, 10) * 1e3}
    return out


def section_tick(torch, dev, scenario, worlds, auto_reset, cores, n=200):
    """Fused tick of another scenario at its BASELINE size + the CPU oracle on the same workload."""
    import numpy as np
    from rl_collision_avoidance_b200.stage_world import StageWorld
    env = StageWorld(BEAMS, scenario=scenario, num_worlds=worlds, device=dev, seed=0, auto_reset=auto_reset)
    env.reset_pose()
    rng = np.random.default_rng(7)
    acts = [torch.from_numpy(random_actions(rng, env.N)).to(dev) for _ in range(16)]
    slots = max(2, int(300e6 / (env.N * BEAMS * 4)) + 1)
    ring = torch.empty(slots, env.N, BEAMS, device=dev)
    def tick(i):
        env.control_vel(acts[i % 16], obs_out=ring[i % slots])
    for i in range(10):
        tick(i)
    torch.cuda.synchronize(dev)
    # like the headline region: the ticks are replayed from a CUDA graph (G even: the state ping-pong closes)
    G = 2 * max(1, min(n, 2 * slots) // 2)
    graph = torch.cuda.CUDAGraph()
    l0 = env.launch_count
    with torch.cuda.graph(graph):
        for i in range(G):
            tick(i)
    launches = (env.launch_count - l0) / G
    graph.replay()
    reps = max(1, n // G)
    ms = gpu_time(torch, dev, lambda i: graph.replay(), reps, warm=1) / G
    N = env.N
    env.close()
    del env, ring
    orc = make_oracle(scenario, worlds, auto_reset=auto_reset)
    orc.reset_world()
    orc.reset_pose()
    ha = [random_actions(rng, orc.N) for _ in range(4)]
    cpu, calls = cpu_sample(lambda i: orc.step(ha[i % 4]), orc.N, cores, seconds=3.0)
    by = N * alg_bytes(BEAMS)
    peak, _ = measured_peak()
    return {'workload': f'{scenario}: {worlds} worlds x {N // worlds} robots = {N} agents, {BEAMS} beams, auto_reset={int(auto_reset)}',
            'us_per_tick': ms * 1e3, 'agent_steps_per_s': N / (ms * 1e-3), 'launches_per_tick': launches,
            'hbm_GBps': by / (ms * 1e-3) / 1e9, 'hbm_frac': by / (ms * 1e-3) / 1e9 / peak,
            'cpu_oracle': {'agent_steps_per_s': cpu, 'cores': cores, 'ticks': calls, 'kind': 'port'}}


def section_sweep(torch, dev, cores):
    """BASELINE config 5: stand-alone raycast at 65 544 robots x {180, 360, 512, 1024} beams; algorithmic bytes
    4*B + 16 per robot (pose in, ranges out)."""
    import numpy as np
    from rl_collision_avoidance_b200.stage_world import StageWorld
    worlds = 2731
    peak, _ = measured_peak()
    rows = []
    for beams in (180, 360, 512, 1024):
        env = StageWorld(beams, scenario='stage1', num_worlds=worlds, device=dev, seed=0, raw_beams=max(512, beams))
        env.reset_pose()
        pose = env.state['pose'].clone()
        slots = max(2, int(300e6 / (env.N * beams * 4)) + 1)
        ring = [torch.empty(env.N, beams, device=dev) for _ in range(slots)]
        ms = gpu_time(torch, dev, lambda i: env.raycast(pose, out=ring[i % slots]), 30, warm=5)
        N = env.N
        by = N * (4 * beams + 16)
        row = {'robots': N, 'beams': beams, 'us': ms * 1e3, 'rays_per_s': N * beams / (ms * 1e-3),
               'hbm_GBps': by / (ms * 1e-3) / 1e9, 'hbm_frac': by / (ms * 1e-3) / 1e9 / peak}
        hp = pose.cpu().numpy()
        env.close()
        del env, ring
        cw = 256                                                   # CPU sample: 256 of the 2731 worlds
        orc = make_oracle('stage1', cw, beams=beams, raw_beams=max(512, beams))
        sub = np.ascontiguousarray(hp[:orc.N])
        cpu, calls = cpu_sample(lambda i: orc.raycast(sub), orc.N * beams, cores, seconds=1.0)
        row['cpu_oracle'] = {'rays_per_s': cpu, 'cores': cores, 'sample': f'{cw} of {worlds} worlds x {calls} sweeps', 'kind': 'port'}
        rows.append(row)
    return rows


def section_train(torch, dev):
    """BASELINE config 2: full PPO on stage 1 — 43 worlds x 24 = 1032 robots, horizon 128, the reference's
    hyper-parameters (ppo_stage1.py:22-35): rollout (policy forward + sampling + tick per step), GAE, 2 epochs of
    1024-row minibatches with an Adam step each.  agent-steps/s over whole updates."""
    from rl_collision_avoidance_b200.model.net import Adam, CNNPolicy
    from rl_collision_avoidance_b200.stage_world import StageWorld
    from rl_collision_avoidance_b200.trainer import run
    env = StageWorld(BEAMS, scenario='stage1', num_worlds=43, device=dev, seed=0, auto_reset=1)
    pol = CNNPolicy(frames=3, action_space=2, device=str(dev), seed=0, max_batch=max(1024, env.N))
    opt = Adam(pol.parameters(), lr=5e-5)
    hp = dict(HORIZON=128, GAMMA=0.99, LAMDA=0.95, BATCH_SIZE=1024, EPOCH=2, COEFF_ENTROPY=5e-4, CLIP_VALUE=0.1,
              NUM_ENV=24, OBS_SIZE=512, ACT_SIZE=2, LASER_HIST=3, MAX_EPISODES=5000)
    import contextlib
    import io
    with contextlib.redirect_stdout(io.StringIO()):
        stats = run(env=env, policy=pol, policy_path=None, action_bound=[[0, -1], [1, 1]], optimizer=opt, hp=hp,
                    stage=1, max_updates=3)
    s = stats[1:]                                               # first update warms up
    roll = sum(x['rollout_s'] for x in s) / len(s)
    upd = sum(x['update_s'] for x in s) / len(s)
    N = env.N
    env.close()
    return {'workload': f'stage1, 43 worlds x 24 = {N} robots, horizon 128, batch 1024, 2 epochs (ppo_stage1.py:22-35)',
            'agent_steps_per_s': 128 * N / (roll + upd), 'rollout_s': roll, 'update_s': upd,
            'rollout_agent_steps_per_s': 128 * N / roll}


def section_circle_dp(torch, dist, dev, rank, world_size, n=100):
    """BASELINE config 4 at N > 1: circle.world, 41 worlds x 50 robots per GPU (16 400 robots at N = 8), worlds sharded
    over the ranks (no data-path collective); graph-replayed ticks, max over ranks.  Its policy-gradient all-reduce is
    the learner_dp section."""
    import numpy as np
    from rl_collision_avoidance_b200.stage_world import StageWorld
    worlds = 41
    err = None
    try:
        env = StageWorld(BEAMS, scenario='circle', num_worlds=worlds, device=dev, seed=0, auto_reset=1,
                         world_offset=rank * worlds)
        env.reset_pose()
        rng = np.random.default_rng(7 + rank)
        acts = [torch.from_numpy(random_actions(rng, env.N)).to(dev) for _ in range(16)]
        slots = max(2, int(300e6 / (env.N * BEAMS * 4)) + 1)
        ring = torch.empty(slots, env.N, BEAMS, device=dev)

        def tick(i):
            env.control_vel(acts[i % 16], obs_out=ring[i % slots])
        for i in range(10):
            tick(i)
        torch.cuda.synchronize(dev)
        G = 2 * max(1, min(n, 2 * slots) // 2)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            for i in range(G):
                tick(i)
        graph.replay()
        torch.cuda.synchronize(dev)
    except Exception as e:                               # every rank must still reach the collectives below
        err = repr(e)
    ok = torch.tensor([0.0 if err else 1.0], device=dev)
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    if float(ok.item()) == 0.0:
        return {'error': err or 'set-up failed on another rank'}
    ms = gpu_time(torch, dev, lambda i: graph.replay(), max(1, n // G), warm=1) / G
    t = torch.tensor([ms], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    N = env.N
    env.close()
    del env, ring
    us = float(t.item()) * 1e3
    return {'workload': f'circle: {world_size} GPUs x {worlds} worlds x 50 robots = {N * world_size} agents, {BEAMS} beams, '
                        'auto_reset=1, worlds sharded over the ranks', 'us_per_tick': us,
            'agent_steps_per_s': N * world_size / (us * 1e-6), 'scaling': 'weak'}


def section_learner_dp(torch, dist, dev, world_size):
    """Data-parallel minibatch step (N > 1): forward + loss + backward + NCCL all-reduce of the flat gradient + Adam
    with the 1/world folded in, at batch 1024 per rank (model/ppo.py:172-188 per optimizer step, SURVEY §8(e))."""
    from rl_collision_avoidance_b200 import _lib
    from rl_collision_avoidance_b200.model.net import Adam, CNNPolicy, _ptr
    pol = CNNPolicy(device=str(dev), max_batch=1024, seed=0)
    opt = Adam(pol.parameters(), lr=5e-5)
    lib, nb = pol.lib, 1024
    obs, gs = torch.rand(nb, 1536, device=dev) - 0.5, torch.rand(nb, 4, device=dev)
    v, mean = torch.empty(nb, device=dev), torch.empty(nb, 2, device=dev)
    act, lp = torch.rand(nb, 2, device=dev), torch.rand(nb, device=dev) - 1
    adv, tgt, losses = torch.randn(nb, device=dev), torch.randn(nb, device=dev), torch.zeros(3, device=dev)
    ws, st = pol._workspace(nb), pol._stream()

    def compute():
        _lib.check(lib.rlca_policy_forward(ws, _ptr(pol.flat), _ptr(obs), _ptr(gs), nb, _ptr(v), _ptr(mean), st))
        _lib.check(lib.rlca_ppo_loss_fwd_bwd(ws, _ptr(pol.flat), _ptr(v), _ptr(mean), _ptr(act), _ptr(lp), _ptr(adv),
                                             _ptr(tgt), nb, 0.1, 5e-4, 20.0, _ptr(losses), st))
        _lib.check(lib.rlca_policy_backward(ws, _ptr(pol.flat), _ptr(obs), _ptr(gs), nb, _ptr(pol.grad), st))

    from rl_collision_avoidance_b200.parallel import OverlappedGradSync
    sync = None

    def full(_=0):                   # RLCA_DP_OVERLAP=1: fc-side ranges all-reduced under the rest of the backward
        compute()
        sync.reduce()
        opt.step(grad_scale=1.0 / world_size)

    def serial(_=0):                 # one all-reduce of the whole buffer after the backward
        compute()
        dist.all_reduce(pol.grad)
        opt.step(grad_scale=1.0 / world_size)

    def local(_=0):
        compute()
        opt.step()

    def ar(_=0):
        dist.all_reduce(pol.grad)

    res = {}
    # the overlapped variant last: while its gradient event is set the backward runs on one stream and leaves 16 SMs to
    # the collective, which must not leak into the other variants
    variants = [('step_serial_allreduce_us', serial), ('step_without_allreduce_us', local), ('allreduce_alone_us', ar),
                ('step_overlapped_allreduce_us', full)]
    for k, fn in variants:
        if fn is full:
            sync = OverlappedGradSync(pol)
        ms = gpu_time(torch, dev, fn, 20, warm=5)
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        res[k] = float(t.item()) * 1e3
    sync.close()
    # the product path: gradient sum + Adam + broadcast as ONE kernel over NVLink peer memory (parallel.PeerAdam)
    try:
        from rl_collision_avoidance_b200.parallel import PeerAdam
        peer = PeerAdam.attach(pol, opt)

        def fused(_=0):
            compute()
            opt.step(grad_scale=1.0 / world_size)

        def fused_alone(_=0):
            opt.step(grad_scale=1.0 / world_size)
        def barriers(_=0):
            peer.hdl.barrier(channel=0)
            peer.hdl.barrier(channel=1)

        def kernel_only(_=0):          # timing only: the two barriers of a real step are what makes it safe
            opt.step_count += 1
            _lib.check(lib.rlca_adam_step_allreduce(peer._grad, peer._param, peer._m, peer._v, peer._mc[0], peer._mc[1],
                                                    peer._mc[2], peer._mc[3], peer.rank, peer.world, peer.n, opt.lr,
                                                    opt.betas[0], opt.betas[1], opt.eps, opt.step_count,
                                                    1.0 / world_size, 0, st))
        for k, fn in (('step_us', fused), ('peer_adam_alone_us', fused_alone), ('peer_barriers_alone_us', barriers),
                      ('peer_kernel_alone_us', kernel_only)):
            ms = gpu_time(torch, dev, fn, 20, warm=5)
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            res[k] = float(t.item()) * 1e3
        res['path'] = 'peer memory, ' + ('NVLS multicast (multimem.ld_reduce / multimem.st)' if peer.nvls else 'P2P loads / stores')
    except Exception as e:
        res['peer_error'] = repr(e)
        res['step_us'] = res['step_serial_allreduce_us']
        res['path'] = 'NCCL all-reduce + Adam'
    res['allreduce_bytes'] = int(pol.flat_size * 4)
    res['collective_share'] = max(0.0, res['step_us'] - res['step_without_allreduce_us']) / res['step_us']
    res['efficiency_vs_no_collective'] = res['step_without_allreduce_us'] / res['step_us']
    res['samples_per_s'] = nb * world_size / (res['step_us'] * 1e-6)
    res['batch_per_rank'] = nb
    res['how'] = ('step_us: forward + loss + backward + ONE kernel that sums the gradient over the ranks, applies Adam and '
                  'writes parameter and moments into every rank (reduce-scatter + Adam + all-gather over peer memory); '
                  'step_serial: NCCL all-reduce of the 8.69 MB buffer + Adam; step_overlapped: fc-side ranges all-reduced '
                  'from a side stream under the rest of the backward')
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=1000)
    ap.add_argument('--warmup', type=int, default=100)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--e2e-steps', type=int, default=200)
    ap.add_argument('--cpu-steps', type=int, default=40)
    ap.add_argument('--e2e-sweep', action='store_true', help='also time step_host for several host-chunk counts')
    ap.add_argument('--ctas-per-world', type=int, default=0)
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--no-graph', action='store_true', help='launch every tick from Python instead of replaying a CUDA graph')
    ap.add_argument('--no-sections', action='store_true', help='skip the extra sections (stage2 / circle / sweep / train / learner)')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help="after the timed ticks, write what the last one returned (rank 0's agents) as DIR/<name>.npy: "
                         'obs, reward, flags, goal_speed, eplog, pose')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get('RANK', '0'))
    world_size = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))

    if args.impl == 'reference':
        if rank != 0:
            return
        from oracle import oracle as orc_mod
        orc_mod.build()                                   # the oracle only: this arm never loads librlca.so
        val, cores, sample, ms = run_cpu(args.steps, args.warmup, budget_s=90.0)
        line = {
            'impl': 'reference', 'metric': METRIC, 'value': val, 'unit': 'agent-steps/s', 'n_gpus': args.gpus,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': WORKLOAD, 'seed': 0,
                       'note': 'reference CPU path = oracle port of Stage semantics; Stage/ROS/mpi4py are not installable here'},
            'cpu_baseline': {'value': val, 'unit': 'agent-steps/s', 'cores': cores, 'kind': 'port', 'sample': sample},
            'e2e': {'value': val, 'unit': 'agent-steps/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0,
        }
        print(json.dumps(line), flush=True)
        return

    import __graft_entry__ as g
    if rank == 0:
        g.build(quiet=True)

    import numpy as np
    import torch
    import torch.distributed as dist
    from rl_collision_avoidance_b200.stage_world import StageWorld

    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world_size > 1:
        dist.init_process_group('nccl', device_id=dev)
        dist.barrier()
    if rank != 0:
        g.build(quiet=True)

    env = StageWorld(BEAMS, index=0, scenario='stage1', num_worlds=WORLDS_PER_GPU, device=dev, seed=0,
                     auto_reset=True, world_offset=rank * WORLDS_PER_GPU, ctas_per_world=args.ctas_per_world)
    env.reset_pose()
    N = env.N
    rng = np.random.default_rng(1000 + rank)
    acts = [torch.from_numpy(random_actions(rng, N)).to(dev) for _ in range(64)]
    # rollout-style obs ring: 128 slots x N x 512 f32 = 1.08 GB > 126 MB L2, so consecutive
    # ticks never re-hit obs lines in L2 (the 0.26 MB simulator state is L2-resident by design)
    ring = torch.empty(128, N, BEAMS, device=dev)

    def tick(i):
        env.control_vel(acts[i % 64], obs_out=ring[i % 128])

    def sync():
        torch.cuda.synchronize(dev)
        if world_size > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    # graph of G consecutive ticks (G even: the state ping-pong returns to its orientation; G divides K)
    G = 0
    if not args.no_graph:
        for cand in range(min(128, args.steps), 15, -1):
            if cand % 2 == 0 and args.steps % cand == 0:
                G = cand
                break
    for i in range(args.warmup):
        tick(i)
    sync()
    graph = None
    launches_per_graph = 0
    if G:
        graph = torch.cuda.CUDAGraph()
        lg = env.launch_count
        with torch.cuda.graph(graph):
            for i in range(G):
                tick(i)
        launches_per_graph = env.launch_count - lg      # kernels captured: physics + lidar per tick
        graph.replay()                                   # untimed: uploads the graph
    sync()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    l0 = env.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sync()
    e0.record()
    if graph is not None:
        for _ in range(args.steps // G):
            graph.replay()
    else:
        for i in range(args.steps):
            tick(i)
    e1.record()
    sync()
    ms = e0.elapsed_time(e1)
    launches = (args.steps // G) * launches_per_graph if graph is not None else env.launch_count - l0
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world_size > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # the last timed tick wrote its scans into the ring slot of its index within the graph (or the loop)
        last = ((G if graph is not None else args.steps) - 1) % 128
        dump_outputs(args.dump_outputs, {'obs': ring[last], 'reward': env.reward, 'flags': env.flags,
                                         'goal_speed': env.gs, 'eplog': env.eplog, 'pose': env.state['pose']})

    # ---- e2e: the host-buffer call (pinned action H2D, tick, obs/reward/flags/gs D2H, sync inside every call)
    a_host = [torch.from_numpy(random_actions(rng, N)).pin_memory() for _ in range(8)]

    def time_e2e(want_obs=True, chunks=0, mode=-1):
        env.set_host_chunks(chunks)
        env.set_host_zero_copy(mode)
        for i in range(5):
            env.step_host(a_host[i % 8], want_obs=want_obs)
        sync()
        t0 = time.perf_counter()
        for i in range(args.e2e_steps):
            env.step_host(a_host[i % 8], want_obs=want_obs)
        torch.cuda.synchronize(dev)
        te = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
        if world_size > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        env.set_host_chunks(0)
        env.set_host_zero_copy(-1)
        return N * world_size * args.e2e_steps / float(te.item())

    e2e_val = time_e2e()                         # library default
    e2e_modes = {'zero_copy_kernel_stores': time_e2e(mode=1), 'dma_serial': time_e2e(chunks=1, mode=0),
                 'dma_2_world_ranges': time_e2e(chunks=2, mode=2)}
    # variant for callers that keep the policy on the device: same call, but the observations stay in HBM
    # (action H2D + tick + reward/flags/goal-speed D2H + sync).  Reported next to `e2e`, never instead of it.
    e2e_noobs = time_e2e(want_obs=False)
    e2e_sweep = None
    if args.e2e_sweep:
        e2e_sweep = {f'mode{m}_chunks{k}': time_e2e(chunks=k, mode=m) for m in (0, 2) for k in (1, 2, 3, 4, 8)}

    learner_dp, circle_dp = None, None
    if world_size > 1 and not args.no_sections:
        try:
            learner_dp = section_learner_dp(torch, dist, dev, world_size)
        except Exception as e:                           # an extra section must not lose the headline line
            learner_dp = {'error': repr(e)}
        try:
            circle_dp = section_circle_dp(torch, dist, dev, rank, world_size)
        except Exception as e:
            circle_dp = {'error': repr(e)}

    if rank == 0:
        value = N * world_size * args.steps / (ms_max * 1e-3)
        per_launch_s = ms_max * 1e-3 / args.steps
        peak, peak_src = measured_peak()
        ach = N * alg_bytes(BEAMS) / per_launch_s / 1e9
        traffic, traffic_src = None, None
        for name in ('r2_step_kernel_traffic.json', 'step_kernel_traffic.json'):
            tp = os.path.join(ROOT, 'profiles', name)
            if os.path.exists(tp):
                try:
                    with open(tp) as f:
                        traffic = json.load(f).get('dram_bytes_per_launch')
                    traffic_src = 'profiles/' + name
                    break
                except Exception:
                    traffic = None
        line = {
            'metric': METRIC, 'value': value, 'unit': 'agent-steps/s', 'n_gpus': world_size, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': ms_max / args.steps, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': WORKLOAD, 'seed': 0,
                       'agents_per_gpu': N, 'beams': BEAMS, 'parallelism': f'worlds sharded over {world_size} GPU(s), '
                       'no data-path collective',
                       'l2': 'obs written round-robin into a 128-slot rollout ring (1.08 GB > 126 MB L2)',
                       'launch': (f'CUDA graph of {G} consecutive ticks replayed {args.steps // G}x ({launches_per_graph // max(G, 1)} kernels per tick: physics, lidar)'
                                  if graph is not None else 'one rlca_env_step call per tick from Python'),
                       'ctas_per_world': args.ctas_per_world or 'auto'},
            'roofline': {'bound': 'hbm', 'achieved': ach, 'peak': peak, 'unit': 'GB/s', 'frac': ach / peak,
                         'traffic': traffic, 'traffic_source': traffic_src, 'peak_source': peak_src,
                         'algorithmic_bytes_per_launch': N * alg_bytes(BEAMS),
                         'note': 'per-GPU; achieved = algorithmic bytes / CUDA-event time per tick over the timed region'},
            'e2e': {'value': e2e_val, 'unit': 'agent-steps/s', 'h2d_bytes_per_step': N * 8 * world_size,
                    'd2h_bytes_per_step': N * (4 * BEAMS + 4 + 4 + 16) * world_size, 'steps': args.e2e_steps,
                    'how': 'rlca_env_step_host with pinned host buffers (library default mode); every call ends with a '
                           'stream synchronize', 'modes': e2e_modes},
            'e2e_obs_on_device': {'value': e2e_noobs, 'unit': 'agent-steps/s', 'h2d_bytes_per_step': N * 8 * world_size,
                                  'd2h_bytes_per_step': N * (4 + 4 + 16) * world_size,
                                  'note': 'same host-buffer call with the scans left in HBM for an on-device policy'},
            'gpu_launches': int(launches),
            'clocks': clocks,
        }
        if e2e_sweep is not None:
            line['e2e_sweep_host_chunks'] = e2e_sweep
        if learner_dp is not None:
            line['learner_dp'] = learner_dp
        if circle_dp is not None:
            line['circle_config4'] = circle_dp
        cores = None
        if world_size == 1 and not args.no_cpu:
            val, cores, sample, _ = run_cpu(args.cpu_steps, 3, budget_s=25.0)
            line['cpu_baseline'] = {'value': val, 'unit': 'agent-steps/s', 'cores': cores, 'kind': 'port',
                                    'sample': sample}
        if world_size == 1:
            line['learner'] = time_learner(dev, N)
        if world_size == 1 and not args.no_sections:
            env.close()
            del ring
            torch.cuda.empty_cache()
            cores = cores or max(1, min(len(os.sched_getaffinity(0)), _cpu_quota() or 10 ** 6))
            sections = {}
            for name, fn in (('learner_reference', lambda: time_learner_reference(dev, N)),
                             ('stage2_tick', lambda: section_tick(torch, dev, 'stage2', 94, 2, cores)),
                             ('circle_tick', lambda: section_tick(torch, dev, 'circle', 41, 1, cores, n=50)),
                             ('raycast_sweep', lambda: section_sweep(torch, dev, cores)),
                             ('train_config2', lambda: section_train(torch, dev))):
                try:
                    sections[name] = fn()
                except Exception as e:                   # an extra section must not lose the headline line
                    sections[name] = {'error': repr(e)}
            line['sections'] = sections
        print(json.dumps(line), flush=True)
    if world_size > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == '__main__':
    main()

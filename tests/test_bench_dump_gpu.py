"""bench.py --steps / --dump-outputs on the headline workload: the number of timed ticks is the one asked for, and the
arrays the last of them returned are written, identical from run to run with the same arguments."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N = 171 * 24


@pytest.mark.parametrize('steps', [40, 17])      # 40: one CUDA graph of 40 ticks; 17: no graph fits, ticks launched one by one
def test_bench_dumps_the_last_timed_tick(built, tmp_path, steps):
    dumps = []
    for run in range(2):
        d = tmp_path / str(run)
        out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', str(steps), '--warmup', '3',
                              '--no-cpu', '--no-sections', '--e2e-steps', '5', '--dump-outputs', str(d)],
                             capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        line = json.loads([l for l in out.stdout.splitlines() if l.strip()][-1])
        assert line['steps'] == steps and line['gpu_launches'] == 2 * steps          # physics + lidar per tick
        dumps.append({p.stem: np.load(p) for p in d.glob('*.npy')})
    a, b = dumps
    assert {k: v.shape for k, v in a.items()} == {'obs': (N, 512), 'reward': (N,), 'flags': (N, 4), 'goal_speed': (N, 4),
                                                  'eplog': (N, 8), 'pose': (N, 4)}
    assert all(v.dtype == np.float32 for v in a.values())
    assert np.all((a['obs'] >= -0.5) & (a['obs'] <= 0.5))                          # scan / 6 - 0.5
    for k in a:
        assert np.array_equal(a[k], b[k]), k

"""The contract of bench.py: the reference arm (the reference forward on the host cores through the oracle port) prints
ONE JSON line with the agreed keys, also under torchrun-style environment variables where only rank 0 may print; the
product arm refuses to run without a GPU instead of falling back; --dump-outputs writes what the last timed step returned."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import rel_err
from fastdepth_b200 import synthetic

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(args, env=None, timeout=600):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py')] + args, capture_output=True, text=True, env=e,
                          timeout=timeout, cwd=ROOT)


def test_reference_arm_line(tmp_path):
    r = run(['--impl', 'reference', '--steps', '1', '--warmup', '1', '--hw', '64', '96', '--dump-outputs', str(tmp_path)])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith('{')]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ('impl', 'metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
              'vs_baseline', 'dtype', 'data', 'config', 'cpu_baseline', 'e2e'):
        assert k in d, k
    assert d['impl'] == 'reference' and d['higher_is_better'] is True and d['value'] > 0 and d['unit'] == 'images/s'
    assert d['cpu_baseline']['kind'] == 'port' and d['cpu_baseline']['cores'] >= 1 and d['cpu_baseline']['value'] == d['value']
    assert d['e2e'] == {'value': d['value'], 'unit': d['unit'], 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
    assert 'workload' in d['config'] and 'model' not in d['config']
    # --dump-outputs: the depth maps of the last timed forward, on the seeded inputs
    from oracle import fastdepth_oracle as orc
    n = d['config']['batch_per_step']
    got = np.load(tmp_path / 'depth.npy')
    assert got.dtype == np.float32 and got.shape == (n, 1, 64, 96)
    want = orc.skipadd_forward(synthetic.synthetic_state_dict(synthetic.STOCK_WIDTHS, seed=1), synthetic.synthetic_input(n, 64, 96, seed=0))
    assert rel_err(torch.from_numpy(got), want) < 1e-5


def test_reference_arm_other_ranks_stay_silent():
    r = run(['--impl', 'reference', '--gpus', '2', '--steps', '1', '--warmup', '1', '--hw', '64', '96'],
            env={'RANK': '1', 'LOCAL_RANK': '1', 'WORLD_SIZE': '2'})
    assert r.returncode == 0 and not [l for l in r.stdout.splitlines() if l.startswith('{')]


@pytest.mark.skipif(torch.cuda.is_available(), reason='checks the no-GPU behaviour')
def test_product_arm_has_no_cpu_fallback():
    r = run(['--steps', '1', '--warmup', '1'])
    assert r.returncode != 0 and 'GPU' in (r.stderr + r.stdout)


@pytest.mark.gpu
def test_product_arm_dumps_its_last_timed_step(tmp_path):
    """--steps 7 over 3 lanes and 4 rotating input batches: the last timed step is the forward of input batch 6 % 4 = 2
    (seed 2), and --dump-outputs must hold exactly what the module's own forward returns for it."""
    import models
    r = run(['--steps', '7', '--warmup', '1', '--batch', '4', '--hw', '64', '96', '--lanes', '3', '--no-eval', '--no-cpu-baseline',
             '--no-lib-baseline', '--e2e-steps', '6', '--stage-iters', '1', '--dump-outputs', str(tmp_path)])
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith('{')][0])
    assert d['steps'] == 7 and d['gpu_launches'] == 7 * d['launches_per_step']
    got = np.load(tmp_path / 'depth.npy')
    assert got.dtype == np.float32 and got.shape == (4, 1, 64, 96)
    m = models.MobileNetSkipAdd((64, 96), pretrained=False, widths=synthetic.STOCK_WIDTHS)
    m.load_state_dict(synthetic.synthetic_state_dict(synthetic.STOCK_WIDTHS, seed=1))
    m = m.eval().cuda().half()
    with torch.no_grad():
        want = m(synthetic.synthetic_input(4, 64, 96, seed=2).cuda().half())
    assert torch.equal(torch.from_numpy(got), want.float().cpu())

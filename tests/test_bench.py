"""bench.py's command line: --steps sets the number of timed steps, --dump-outputs writes what the timed path returned."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BENCH = os.path.join(ROOT, 'bench.py')


def _bench(*args):
    return subprocess.run([sys.executable, BENCH, *args], capture_output=True, text=True, cwd=ROOT, timeout=900)


@pytest.mark.parametrize('args,msg', [(('--steps', '0'), '--steps must be at least 1'),
                                      (('--impl', 'reference', '--dump-outputs', 'x'), '--dump-outputs applies to --impl ours')])
def test_rejected_arguments(args, msg):
    out = _bench(*args)
    assert out.returncode == 2 and msg in out.stderr, out.stderr


@pytest.mark.gpu
def test_steps_and_dump_outputs(tmp_path):
    out = _bench('--gpus', '1', '--steps', '2', '--warmup', '1', '--no-extras', '--dump-outputs', str(tmp_path))
    assert out.returncode == 0, out.stderr[-3000:]
    res = json.loads(out.stdout.strip().splitlines()[-1])
    assert res['steps'] == 2 and res['launch_counts']['loss_single_pass'] == 2, res
    assert sorted(os.listdir(tmp_path)) == ['grad.npy', 'grad_corners.npy', 'loss.npy']
    assert sum(os.path.getsize(tmp_path / n) for n in os.listdir(tmp_path)) <= 64 << 20
    loss, grad, corners = (np.load(tmp_path / n) for n in ('loss.npy', 'grad.npy', 'grad_corners.npy'))
    assert loss.dtype == grad.dtype == corners.dtype == np.float32
    assert loss.shape == (4,) and corners.shape == (2, 512, 512) and 4_000_000 < grad.size <= 1 << 22
    assert np.isfinite(loss).all() and np.isfinite(grad).all() and np.isfinite(corners).all()
    assert abs(loss[:3].sum() - loss[3]) <= 1e-6 * abs(loss[3])
    assert np.abs(grad).max() > 0

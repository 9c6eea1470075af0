"""bench.py --dump-outputs: the last timed step's gradient buffer and weights, identical for identical arguments, and --steps sets how
many steps ran before them."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir, steps):
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--config', 'cfg1', '--steps', str(steps), '--warmup', '3',
                          '--e2e-steps', '1', '--no-cpu-baseline', '--no-extras', '--dump-outputs', str(out_dir)],
                         capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith('{')][-1])
    assert line['steps'] == steps
    return line, {k: np.load(os.path.join(out_dir, k + '.npy')) for k in ('grad_buffer', 'weights')}


def test_dump_outputs_are_reproducible_and_follow_steps(tmp_path):
    line, a = _bench(tmp_path / 'a', 2)
    _, b = _bench(tmp_path / 'b', 2)
    _, c = _bench(tmp_path / 'c', 3)
    n = len(a['weights'])
    assert a['grad_buffer'].dtype == np.float32 and a['weights'].dtype == np.float32
    assert a['grad_buffer'].shape == (n + 2,)
    assert a['grad_buffer'][n + 1] == line['config']['per_gpu_batch']          # mask count of one step over the whole batch
    assert np.isfinite(a['grad_buffer']).all() and np.isfinite(a['weights']).all()
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    assert not np.array_equal(a['weights'], c['weights'])

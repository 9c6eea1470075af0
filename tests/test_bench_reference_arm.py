"""bench.py --impl reference (the CPU arm that is run beside ours) needs no GPU: run it on the default 400-node workload and
check the JSON line carries the keys every bench line has, and the outputs --dump-outputs writes."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--config', 'cfg1', '--steps', '1',
                          '--warmup', '1', '--dump-outputs', str(tmp_path)], capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith('{')]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and d['gpu_launches'] == 0
    for key in ('metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling', 'vs_baseline',
                'dtype', 'data', 'config', 'cpu_baseline', 'e2e'):
        assert key in d, key
    assert d['unit'] == 'trajectories/s' and d['value'] > 0 and d['higher_is_better'] is True
    assert d['cpu_baseline']['kind'] in ('port', 'reference') and d['cpu_baseline']['cores'] >= 1 and d['cpu_baseline']['value'] == d['value']
    assert d['e2e'] == {'value': d['value'], 'unit': d['unit'], 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
    assert 'workload' in d['config'] and 'model' not in d['config']
    buf = np.load(os.path.join(str(tmp_path), 'grad_buffer.npy'))            # [grads | nll_sum | count] of the sampled trajectories
    n = d['config']['sample_trajectories_per_step']
    assert buf.dtype == np.float32 and buf[-1] == n and buf[-2] > 0 and np.isfinite(buf).all()
    assert sorted(os.listdir(str(tmp_path))) == ['grad_buffer.npy']                # no optimizer step, so no weights

"""Data-parallel training in the product API on real hardware (SURVEY 4 iv): 2 ranks (torchrun, one GPU each) against the
1-GPU run of the same script — the summed gradient buffer and the weights after 3 epochs of Scone_GCN.train — with both exchanges:
the library's NVLink peer-memory kernel fused with Adam (default) and the NCCL all-reduce."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason='needs 2 GPUs')
@pytest.mark.parametrize('exchange', ['peer', 'nccl'])
def test_two_gpu_training_matches_one_gpu(tmp_path, exchange):
    one, two = str(tmp_path / 'one.npz'), str(tmp_path / 'two.npz')
    env = dict(os.environ)
    env.pop('WORLD_SIZE', None)
    env['SCONE_DP_EXCHANGE'] = exchange
    subprocess.check_call([sys.executable, os.path.join(HERE, 'dp_worker.py'), one], env=env, timeout=600)
    port = 29600 + os.getpid() % 1000
    subprocess.check_call([sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2', '--master-addr', '127.0.0.1',
                           '--master-port', str(port), os.path.join(HERE, 'dp_worker.py'), two], env=env, timeout=900)
    a, b = np.load(one), np.load(two)
    assert int(a['world']) == 1 and int(b['world']) == 2
    assert bool(b['ident'])                                             # peer exchange: bit-identical weights on both ranks
    n = len(a['grads']) - 2
    assert a['grads'][n + 1] == b['grads'][n + 1]                       # mask count: exact
    assert abs(a['grads'][n] - b['grads'][n]) <= 1e-6 * abs(a['grads'][n])
    # fixed-order sums inside each rank, one sum over ranks: equal up to the grouping of the fp32 sums
    assert np.abs(a['grads'][:n] - b['grads'][:n]).max() <= 1e-5 * np.abs(a['grads'][:n]).max()
    for i in range(10):
        assert np.abs(a['w%d' % i] - b['w%d' % i]).max() <= 1e-5 * max(1.0, np.abs(a['w%d' % i]).max())
    assert np.allclose(a['result'], b['result'], rtol=1e-5, atol=1e-6)

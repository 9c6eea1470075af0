"""Data-parallel host logic on CPU: 2 gloo ranks shard the batch, all-reduce [grads | nll | count], and must agree with
the single-process result (oracle arithmetic; the CUDA kernels play no part here)."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from golden_util import Dataset, load, weights_of
from scone_gcn_b200.dp import allreduce_sum_, shard_range


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from oracle import scone_oracle as so
    dist.init_process_group('gloo', rank=rank, world_size=world)
    ds = Dataset('dataset_small.npz')
    fx = load('model_small_scone_h16.npz')
    W = weights_of(fx, 'w_big')
    te = np.stack([np.nonzero(ds.B2[:, f])[0] for f in range(ds.F)])
    ts = np.stack([ds.B2[te[f], f] for f in range(ds.F)])
    orc = so.SparseOracle('scone', ds.edges, te, ts, ds.N, dtype=np.float64)
    lo, hi = shard_range(ds.n_traj, rank, world)
    X = ds.flows[lo:hi, :, 0].T.copy()
    mask = ds.train_mask[lo:hi].astype(np.float64)
    nll, g = orc.loss_and_grads(W, X, ds.last_nodes[lo:hi], ds.raw['targets_argmax'][lo:hi], mask)
    buf = torch.from_numpy(np.concatenate([x.ravel() for x in g] + [np.array([nll, mask.sum()])]))
    allreduce_sum_(buf)
    if rank == 0:
        np.save(out, buf.numpy())
    dist.destroy_process_group()


def test_shard_range_partitions():
    for n in (0, 1, 7, 60, 4096):
        for w in (1, 2, 3, 8):
            spans = [shard_range(n, r, w) for r in range(w)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            assert max(h - l for l, h in spans) - min(h - l for l, h in spans) <= 1


def test_two_rank_allreduce_matches_single_process(tmp_path):
    from oracle import scone_oracle as so
    out = str(tmp_path / 'buf.npy')
    port = 29500 + os.getpid() % 2000
    mp.spawn(_worker, args=(2, port, out), nprocs=2, join=True)
    got = np.load(out)
    ds = Dataset('dataset_small.npz')
    fx = load('model_small_scone_h16.npz')
    W = weights_of(fx, 'w_big')
    te = np.stack([np.nonzero(ds.B2[:, f])[0] for f in range(ds.F)])
    ts = np.stack([ds.B2[te[f], f] for f in range(ds.F)])
    orc = so.SparseOracle('scone', ds.edges, te, ts, ds.N, dtype=np.float64)
    mask = ds.train_mask.astype(np.float64)
    nll, g = orc.loss_and_grads(W, ds.flows[:, :, 0].T.copy(), ds.last_nodes, ds.raw['targets_argmax'], mask)
    ref = np.concatenate([x.ravel() for x in g] + [np.array([nll, mask.sum()])])
    assert np.allclose(got, ref, rtol=1e-10, atol=1e-12)


def _shard_worker(rank, world, port, out):
    # no visible GPU: dp.init_from_env would otherwise take NCCL with one GPU per rank, and this test is about the gloo path
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), CUDA_VISIBLE_DEVICES='')
    from scone_gcn_b200 import dp
    assert dp.init_from_env() == (rank, world) and dp.is_distributed()
    rows = np.arange(100, 137)                              # the batch rows every rank derives from the shared RNG stream
    mine = dp.shard_rows(rows)
    t = torch.zeros(137, dtype=torch.float64)
    t[mine] = 1.0
    dp.allreduce_sum_(t)                                    # every row owned exactly once
    if rank == 0:
        np.save(out, t.numpy())
    dist.destroy_process_group()


def test_product_sharding_covers_every_batch_row_once(tmp_path):
    """Scone_GCN.train shards each batch with dp.shard_rows and all-reduces with dp.allreduce_sum_ (world_size 2, gloo)."""
    out = str(tmp_path / 'own.npy')
    port = 31500 + os.getpid() % 2000
    mp.spawn(_shard_worker, args=(2, port, out), nprocs=2, join=True)
    own = np.load(out)
    assert np.array_equal(own[100:137], np.ones(37)) and own[:100].sum() == 0

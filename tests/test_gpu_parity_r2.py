"""Round-2 parity cases (VERDICT r1, items 1-2): the CUDA path against the ORACLE on the shapes the bench runs (hidden 32 on a
large sparse complex), with `-flip_edges`, and for ebli / mixed widths — all through the C ABI (ctypes), north-star
tolerances: log-probs 1e-5, gradients 1e-4 (relative to the largest entry)."""
import numpy as np
import pytest
import torch

from golden_util import Dataset
from oracle import scone_oracle as so

pytestmark = pytest.mark.gpu


def _sparse_problem(n_nodes, n_traj, seed):
    from scone_gcn_b200 import synthetic_data_gen as sdg
    from scone_gcn_b200.complex import incidence_lists_from_simplices
    sp = sdg.generate_sparse_dataset(n_nodes, n_traj, seed=seed, n_waypoints=24)
    en, es, te, ts = incidence_lists_from_simplices(sp.edges, sp.faces)
    return sp, te, ts


def _dense_X(sp, B):
    X = np.zeros((len(sp.edges), B), np.float32)
    for t in range(B):
        sl = slice(sp.traj_ptr[t], sp.traj_ptr[t + 1])
        X[sp.flow_edge[sl], t] = sp.flow_val[sl]
    return X


def check_against_sparse_oracle(net, sp, te, ts, model, W, B, dtype, lp_tol=1e-5, g_tol=1e-4):
    """log-probs + NLL + gradients of the first B trajectories of `sp`, CUDA path vs SparseOracle(dtype)."""
    nnz = int(sp.traj_ptr[B])
    ptr, fe, fv = sp.traj_ptr[:B + 1], sp.flow_edge[:nnz], sp.flow_val[:nnz]
    last, tgt = sp.last_nodes[:B], sp.target_idx[:B]
    mask = np.ones(B, np.float32)
    mask[B // 3] = 0.0
    orc = so.SparseOracle(model, sp.edges, te, ts, int(sp.n_nodes), dtype=dtype)
    X = _dense_X(sp, B)
    lp_ref = orc.forward(W, X, last)
    lp = net.forward(ptr, fe, fv, last)
    D = min(lp.shape[1], lp_ref.shape[1])
    assert lp.shape[1] == lp_ref.shape[1]
    err = np.abs(lp[:, :D] - lp_ref[:, :D]).max()
    assert err <= lp_tol * max(1.0, np.abs(lp_ref).max()), err
    nll_ref, g_ref = orc.loss_and_grads(W, X, last, tgt, mask)
    buf = net.loss_grad(ptr, fe, fv, last, tgt, mask)
    k = net.n_params
    assert buf[k + 1] == mask.sum()
    assert abs(buf[k] - nll_ref) <= 1e-5 * max(1.0, abs(nll_ref)) * B
    grads = net.unflatten(buf[:k])
    for a, r in zip(grads, g_ref):
        assert np.abs(a - r).max() <= g_tol * max(np.abs(r).max(), 1e-30), (a.shape, np.abs(a - r).max(), np.abs(r).max())
    return err


@pytest.mark.parametrize('dtype,B', [(np.float32, 64), (np.float64, 16)])
def test_hidden32_on_50k_node_complex_vs_sparse_oracle(dtype, B):
    """The benchmarked shape (cfg4 / cfg5: hidden 32, large sparse holed Delaunay complex from generate_sparse_dataset) against the
    oracle: the default model-level pipeline vs SparseOracle in fp32 and its fp64 twin."""
    import scone_gcn_b200 as sg
    sp, te, ts = _sparse_problem(50000, 64, seed=7)
    cx = sg.SimplicialComplex.from_simplices(int(sp.n_nodes), sp.edges, sp.faces, 'scone')
    net = sg.SconeModel(cx, [32, 32, 32], micro_batch=48)                 # ragged second micro-batch at B = 64
    rs = np.random.RandomState(3)
    W = [0.3 * rs.randn(*s) for s in net.shapes]
    net.set_weights(W)
    check_against_sparse_oracle(net, sp, te, ts, 'scone', W, B, dtype)


def test_ebli_hidden32_on_sparse_complex_vs_sparse_oracle():
    import scone_gcn_b200 as sg
    sp, te, ts = _sparse_problem(3000, 24, seed=11)
    cx = sg.SimplicialComplex.from_simplices(int(sp.n_nodes), sp.edges, sp.faces, 'ebli')
    net = sg.SconeModel(cx, [32, 32, 32], micro_batch=16)
    rs = np.random.RandomState(5)
    W = [0.05 * rs.randn(*s) for s in net.shapes]                        # L1^2 has entries up to ~30: keep activations O(1)
    net.set_weights(W)
    check_against_sparse_oracle(net, sp, te, ts, 'ebli', W, 24, np.float64)


@pytest.mark.parametrize('model,hidden,scale', [('ebli', [32, 32, 32], 0.05), ('scone', [16, 32, 16], 0.3), ('ebli', [32, 16], 0.05),
                                                ('scone', [32], 0.3), ('scone', [8, 8, 8], 0.4), ('scone', [64, 64, 64], 0.15),
                                                ('scone', [8, 16, 32], 0.3), ('ebli', [64, 32, 16], 0.03), ('scone', [32, 64], 0.2),
                                                ('scone', [8], 0.4), ('scone', [64], 0.2), ('scone', [16, 16, 16, 16], 0.3),
                                                ('scone', [32, 32, 32, 32, 32], 0.2)])
def test_widths_and_depths_vs_dense_oracle(model, hidden, scale):
    """ebli h32, mixed widths (ratio-2 chains through 8 and 64), widths 8 and 64, 1- and 2-layer nets and nets deeper than 3 layers
    against the DENSE oracle (the reference formulation) on the small complex, on the pipeline each starts on: widths 8 / 64 only run
    on the unit kernels (0) and every other pipeline refuses them; more than 3 layers or mixed widths are not fused and start on the
    cone pipeline (3, D = 9 here); uniform 16 / 32 with at most 3 layers start fused (4)."""
    import scone_gcn_b200 as sg
    from scone_gcn_b200._lib import SconeError
    ds = Dataset('dataset_small.npz')
    cx = sg.SimplicialComplex.from_dense(ds.B1, ds.B2, model)
    net = sg.SconeModel(cx, hidden, micro_batch=40)
    if any(c in (8, 64) for c in hidden):
        assert net.pipeline == 0
        for which in (1, 2, 3, 4):
            with pytest.raises(SconeError):
                net.set_pipeline(which)
        assert net.pipeline == 0
    else:
        assert net.pipeline == (4 if len(set(hidden)) == 1 and len(hidden) <= 3 else 3)
    rs = np.random.RandomState(9)
    W = [scale * rs.randn(*s) for s in net.shapes]
    net.set_weights(W)
    ptr, fe, fv = sg.flows_to_csr(ds.flows)
    lp = net.forward(ptr, fe, fv, ds.last_nodes)
    orc = so.DenseOracle(model, so.shift_matrices(ds.B1, ds.B2, model), ds.B1, ds.last_nodes, ds.flows, ds.targets, dtype=torch.float64)
    with torch.no_grad():
        ref = orc.forward(W).numpy()[:, :, 0]
    assert np.abs(lp - ref).max() <= 1e-5 * max(1.0, np.abs(ref).max())
    mask = ds.train_mask.astype(np.float32)
    buf = net.loss_grad(ptr, fe, fv, ds.last_nodes, ds.raw['targets_argmax'], mask)
    k = net.n_params
    _, g_ref = orc.loss_and_grads(W, ds.train_mask, 0.0)
    for a, r in zip(net.unflatten(buf[:k] / buf[k + 1]), g_ref):
        assert np.abs(a - r).max() <= 1e-4 * max(np.abs(r).max(), 1e-30)


@pytest.mark.parametrize('model', ['scone', 'ebli'])
def test_flip_edges_vs_dense_oracle(model):
    """`-flip_edges 1` (trajectory_experiments.py:214-219,242-244,290-296): F L F shifts, B1_jax F readout, X F flows, with the
    reference's own draw of F (seed 1, p = [0.8, 0.2])."""
    import scone_gcn_b200 as sg
    ds = Dataset('dataset_small.npz')
    np.random.seed(1)
    flips = np.random.choice([1, -1], size=ds.E, replace=True, p=[0.8, 0.2])
    assert (flips == -1).sum() > 0
    cx = sg.SimplicialComplex.from_dense(ds.B1, ds.B2, model, flips=flips)
    shifts = so.shift_matrices(ds.B1, ds.B2, model, flips=flips)
    for k in range(2):                                                    # integer work: bit-exact
        assert np.array_equal(cx.shift_dense(k), np.asarray(shifts[k]))
    flows = ds.flows * flips[None, :, None]
    net = sg.SconeModel(cx, [16, 16, 16], micro_batch=64)
    rs = np.random.RandomState(4)
    W = [(0.3 if model == 'scone' else 0.05) * rs.randn(*s) for s in net.shapes]
    net.set_weights(W)
    ptr, fe, fv = sg.flows_to_csr(flows)
    lp = net.forward(ptr, fe, fv, ds.last_nodes)
    orc = so.DenseOracle(model, shifts, ds.B1 @ np.diag(flips), ds.last_nodes, flows, ds.targets, dtype=torch.float64)
    with torch.no_grad():
        ref = orc.forward(W).numpy()[:, :, 0]
    assert np.abs(lp - ref).max() <= 1e-5 * max(1.0, np.abs(ref).max())
    mask = ds.train_mask.astype(np.float32)
    buf = net.loss_grad(ptr, fe, fv, ds.last_nodes, ds.raw['targets_argmax'], mask)
    k = net.n_params
    _, g_ref = orc.loss_and_grads(W, ds.train_mask, 0.0)
    for a, r in zip(net.unflatten(buf[:k] / buf[k + 1]), g_ref):
        assert np.abs(a - r).max() <= 1e-4 * max(np.abs(r).max(), 1e-30)

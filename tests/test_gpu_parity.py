"""GPU parity tests: the CUDA path (through the C ABI) against the oracle and the golden fixtures.

Tolerances are the north-star's: integer/index work bit-exact; log-probs within 1e-5, gradients within
1e-4 (relative to the largest magnitude of the tensor), identical next-node accuracy.
"""
import numpy as np
import pytest
import torch

from golden_util import Dataset, load, weights_of
from oracle import scone_oracle as so

pytestmark = pytest.mark.gpu

LP_TOL = 1e-5
GRAD_TOL = 1e-4


def _mods():
    import scone_gcn_b200 as sg
    return sg


def _relmax(a, b):
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


@pytest.fixture(scope='module')
def small():
    return Dataset('dataset_small.npz')


@pytest.mark.parametrize('model', ['scone', 'ebli'])
def test_index_arrays_bit_exact_on_device_handle(small, model):
    sg = _mods()
    cx = sg.SimplicialComplex.from_dense(small.B1, small.B2, model)
    ref = so.shift_matrices(small.B1, small.B2, model)
    for k in range(2):
        assert np.array_equal(cx.shift_dense(k), ref[k])
    nb, _, _ = so.neighbourhood_tables(small.B1, small.last_nodes)
    assert np.array_equal(cx.nbrhoods, nb)


@pytest.mark.parametrize('name,mb', [('model_small_scone_h16', 64), ('model_small_scone_h16', 7),
                                     ('model_small_ebli_h16', 64), ('model_small_scone_h32', 16)])
def test_forward_and_grads_vs_reference_golden(small, name, mb):
    sg = _mods()
    fx = load(name + '.npz')
    model = str(fx['model'])
    hidden = [int(h[1]) for h in fx['hidden']]
    cx = sg.SimplicialComplex.from_dense(small.B1, small.B2, model)
    net = sg.SconeModel(cx, hidden, micro_batch=mb)
    ptr, fe, fv = sg.flows_to_csr(small.flows)
    tgt = small.raw['targets_argmax']
    mask = fx['batch_mask'].astype(np.float32)
    wd = float(fx['wd'])
    for tag in ('init', 'big'):
        W = weights_of(fx, 'w_' + tag)
        net.set_weights(W)
        lp = net.forward(ptr, fe, fv, small.last_nodes)
        ref = fx[tag + '_logprobs'][:, :, 0]
        assert np.abs(lp - ref).max() <= LP_TOL * max(1.0, np.abs(ref).max()), (tag, np.abs(lp - ref).max())
        buf = net.loss_grad(ptr, fe, fv, small.last_nodes, tgt, mask)
        n = net.n_params
        count = buf[n + 1]
        assert count == mask.sum()
        ridge = wd * sum(float((np.asarray(w, np.float64) ** 2).sum()) for w in W)
        loss = buf[n] / count + ridge
        assert loss == pytest.approx(float(fx[tag + '_loss_batch']), rel=2e-5)
        grads = net.unflatten(buf[:n] / count)
        for i, g in enumerate(grads):
            g = g + 2 * wd * np.asarray(W[i], np.float32)
            r = fx['%s_grad_%d' % (tag, i)]
            assert _relmax(g, r) <= GRAD_TOL, (tag, i, _relmax(g, r))
        # identical next-node accuracy (scone_trajectory_model.py:59-71)
        pred = lp.copy()
        nn = fx['n_nbrs']
        for i in range(len(pred)):
            pred[i, nn[i]:] = -100
        for mname, m in (('train', small.train_mask), ('test', small.test_mask)):
            acc = np.mean(np.argmax(pred[m == 1], axis=1) == tgt[m == 1])
            assert acc == pytest.approx(float(fx['%s_acc_%s' % (tag, mname)]), abs=1e-7)


def test_deterministic_and_microbatch_invariant_logprobs(small):
    sg = _mods()
    fx = load('model_small_scone_h16.npz')
    cx = sg.SimplicialComplex.from_dense(small.B1, small.B2, 'scone')
    ptr, fe, fv = sg.flows_to_csr(small.flows)
    W = weights_of(fx, 'w_big')
    outs, grads = [], []
    for mb in (64, 64, 5):
        net = sg.SconeModel(cx, [16, 16, 16], micro_batch=mb)
        net.set_weights(W)
        outs.append(net.forward(ptr, fe, fv, small.last_nodes))
        grads.append(net.loss_grad(ptr, fe, fv, small.last_nodes, small.raw['targets_argmax'],
                                   np.ones(small.n_traj, np.float32)))
    assert np.array_equal(outs[0], outs[1]) and np.array_equal(grads[0], grads[1])       # run-to-run bit-exact
    assert np.array_equal(outs[0], outs[2])            # per-trajectory results do not depend on the micro-batch
    assert _relmax(grads[2], grads[0]) < 1e-5


def test_row_ids_beyond_2_31_microbatch_invariant():
    """Maximum sizes: ONE micro-batch whose trajectory-major row ids t*E + e run past 2^31 (E * micro_batch in (2^31, 2^32), the
    cfg5 bench shape) against the same trajectories in micro-batches of 1024.  The batch tiles 256 generated trajectories, so
    every tile must reproduce the first one bit for bit; gradients agree within fp32 summation noise."""
    sg = _mods()
    from scone_gcn_b200 import synthetic_data_gen as sdg
    sp = sdg.generate_sparse_dataset(50000, 256, seed=7, n_waypoints=8)
    cx = sg.SimplicialComplex.from_simplices(int(sp.n_nodes), sp.edges, sp.faces, 'scone')
    base = 256
    tiles = int(2.25e9 // cx.E) // base + 1
    B = tiles * base
    assert (1 << 31) < cx.E * B < (1 << 32)
    nnz = int(sp.traj_ptr[base])
    ptr = np.concatenate([[0], np.cumsum(np.tile(np.diff(sp.traj_ptr[:base + 1]), tiles))]).astype(np.int32)
    fe = np.tile(sp.flow_edge[:nnz], tiles).astype(np.int32)
    fv = np.tile(sp.flow_val[:nnz], tiles).astype(np.float32)
    last = np.tile(sp.last_nodes[:base], tiles).astype(np.int32)
    tgt = np.tile(sp.target_idx[:base], tiles).astype(np.int32)
    rs = np.random.RandomState(3)
    mask = (rs.rand(B) < 0.8).astype(np.float32)
    res = []
    for mb in (B, 1024):
        net = sg.SconeModel(cx, [16, 16, 16], micro_batch=mb)
        if mb == B:
            rs_w = np.random.RandomState(11)
            W = [0.2 * rs_w.randn(*s_) for s_ in net.shapes]
        net.set_weights(W)
        lp = net.forward(ptr, fe, fv, last)
        buf = net.loss_grad(ptr, fe, fv, last, tgt, mask)
        res.append((lp, buf))
        del net
        torch.cuda.empty_cache()
    lp_big, lp_small = res[0][0], res[1][0]
    assert np.isfinite(lp_big).all() and np.abs(lp_big).max() > 0
    assert np.array_equal(lp_big, lp_small)
    assert np.array_equal(lp_big.reshape(tiles, base, -1), np.broadcast_to(lp_big[:base], (tiles, base, lp_big.shape[1])))
    n = len(res[0][1]) - 2
    assert res[0][1][n + 1] == res[1][1][n + 1] == mask.sum()
    assert _relmax(res[0][1][:n + 1], res[1][1][:n + 1]) < 1e-4


@pytest.mark.parametrize('scale', [0.0, 0.3])
def test_device_accuracy_matches_numpy(small, scale):
    """Evaluation on the device (SURVEY 8f.3): forward + mask-to--100 + argmax + compare (scone_trajectory_model.py:59-71) against
    the same steps in NumPy on the returned log-probs — integer counts, exact; scale 0 = all log-probs tie (first maximum)."""
    sg = _mods()
    from scone_gcn_b200.scone_trajectory_model import Scone_GCN
    cx = sg.SimplicialComplex.from_dense(small.B1, small.B2, 'scone')
    ptr, fe, fv = sg.flows_to_csr(small.flows)
    net = sg.SconeModel(cx, [16, 16, 16], micro_batch=13)
    rs = np.random.RandomState(4)
    net.set_weights([scale * rs.randn(*s_) for s_ in net.shapes])
    _, n_nbrs, _ = so.neighbourhood_tables(small.B1, small.last_nodes)
    tgt = small.raw['targets_argmax']
    for mask in (np.ones(small.n_traj, np.float32), (rs.rand(small.n_traj) < 0.5).astype(np.float32)):
        lp = net.forward(ptr, fe, fv, small.last_nodes)
        ref = Scone_GCN._accuracy_from(lp[:, :, None], tgt[mask == 1][:, None], mask, n_nbrs)     # [n, 1] like argmax(y[mask == 1], axis=1)
        correct, counted = net.accuracy(ptr, fe, fv, small.last_nodes, n_nbrs, tgt, mask)
        assert counted == int(mask.sum())
        assert correct / counted == ref
    # fewer valid slots than the true degree: the -100 masking decides
    half = np.maximum(1, np.asarray(n_nbrs) // 2)
    mask = np.ones(small.n_traj, np.float32)
    ref = Scone_GCN._accuracy_from(net.forward(ptr, fe, fv, small.last_nodes)[:, :, None], tgt[:, None], mask, half)
    correct, counted = net.accuracy(ptr, fe, fv, small.last_nodes, half, tgt, mask)
    assert correct / counted == ref


def test_default_complex_vs_reference_golden():
    sg = _mods()
    ds = Dataset('dataset_default.npz')
    fx = load('model_default_scone_h16.npz')
    cx = sg.SimplicialComplex.from_simplices(ds.N, ds.edges, ds.faces, 'scone')
    assert (cx.N, cx.E, cx.F, cx.D) == (400, 1001, 649, 13)
    net = sg.SconeModel(cx, [16, 16, 16], micro_batch=256)
    ptr, fe, fv = sg.flows_to_csr(ds.flows)
    tgt = ds.raw['targets_argmax']
    mask = fx['batch_mask'].astype(np.float32)
    for tag in ('init', 'big'):
        W = weights_of(fx, 'w_' + tag)
        net.set_weights(W)
        lp = net.forward(ptr, fe, fv, ds.last_nodes)
        ref = fx[tag + '_logprobs'][:, :, 0]
        assert np.abs(lp - ref).max() <= LP_TOL * max(1.0, np.abs(ref).max())
        buf = net.loss_grad(ptr, fe, fv, ds.last_nodes, tgt, mask)
        n = net.n_params
        grads = net.unflatten(buf[:n] / buf[n + 1])
        for i, g in enumerate(grads):
            g = g + 2 * float(fx['wd']) * np.asarray(W[i], np.float32)
            assert _relmax(g, fx['%s_grad_%d' % (tag, i)]) <= GRAD_TOL, (tag, i)
    assert float(fx['init_loss_train']) == pytest.approx(np.log(13), abs=1e-3)


@pytest.mark.parametrize('cin,cout,act', [(16, 16, 0), (32, 32, 0), (8, 8, 1), (16, 32, 0), (32, 16, 2), (64, 64, 0),
                                          (1, 16, 0), (1, 32, 1)])
@pytest.mark.parametrize('b', [5, 32])
def test_layer_kernels_dense_random_input(small, cin, cout, act, b):
    """Kernel-level: one fused layer forward/backward on DENSE random features (no structural zeros)."""
    sg = _mods()
    from scone_gcn_b200 import _lib
    L = _lib.lib()
    cx = sg.SimplicialComplex.from_dense(small.B1, small.B2, 'scone')
    E = cx.E
    rs = np.random.RandomState(cin * 100 + cout + b)
    Hin = rs.randn(E, b, cin).astype(np.float32)
    W = [(rs.randn(cin, cout) * 0.3).astype(np.float32) for _ in range(3)]
    G = rs.randn(E, b, cout).astype(np.float32)
    S = [cx.shift_dense(0), cx.shift_dense(1)]
    # fp64 reference
    H64 = Hin.astype(np.float64)
    T = [H64, np.einsum('ef,fbc->ebc', S[0], H64), np.einsum('ef,fbc->ebc', S[1], H64)]
    Z = sum(T[k] @ W[k].astype(np.float64) for k in range(3))
    actf = [np.tanh, lambda z: np.where(z >= 0, z, 0.01 * z), lambda z: np.maximum(z, 0)][act]
    dact = [lambda h: 1 - h * h, lambda h: np.where(h >= 0, 1.0, 0.01), lambda h: (h > 0) * 1.0][act]
    Href = actf(Z)
    dev = torch.device('cuda')
    rank = torch.from_numpy(cx.edge_rank.astype(np.int64))          # caller's edge id -> internal device row

    def to_dev(a):                                                   # rows in the library's internal order
        t = torch.empty(a.shape, dtype=torch.float32)
        t[rank] = torch.from_numpy(a)
        return t.to(dev)

    def from_dev(t):
        return t.cpu()[rank].numpy()
    tH, tG = to_dev(Hin), to_dev(G)
    tW = [torch.from_numpy(w).to(dev) for w in W]
    tout = torch.empty(E, b, cout, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    _lib.check(L.scone_layer_forward(cx.handle, act, b, cin, cout, _lib.dptr(tH), _lib.dptr(tW[0]), _lib.dptr(tW[1]),
                                     _lib.dptr(tW[2]), _lib.dptr(tout), None, None, None, st), 'layer_forward')
    out = from_dev(tout)
    assert np.abs(out - Href).max() <= 2e-5 * max(1.0, np.abs(Href).max())
    # backward: G is dL/dZ
    G64 = G.astype(np.float64)
    A = [G64, np.einsum('ef,fbc->ebc', S[0], G64), np.einsum('ef,fbc->ebc', S[1], G64)]
    dW_ref = np.stack([np.einsum('ebi,ebo->io', H64, A[k]) for k in range(3)])
    ws = torch.empty(L.scone_layer_backward_workspace_bytes(cin, cout) // 4 + 16, device=dev)
    tdW = torch.zeros(3, cin, cout, device=dev)
    tGp = torch.empty(E, b, cin, device=dev) if cin > 1 else None
    _lib.check(L.scone_layer_backward(cx.handle, act, b, cin, cout, _lib.dptr(tG), _lib.dptr(tH), _lib.dptr(tW[0]),
                                      _lib.dptr(tW[1]), _lib.dptr(tW[2]), _lib.dptr(tGp), _lib.dptr(tdW), 0, _lib.dptr(ws),
                                      None, None, None, None, st), 'layer_backward')
    assert _relmax(tdW.cpu().numpy(), dW_ref) <= 2e-5
    if cin > 1:
        dH = sum(A[k] @ W[k].astype(np.float64).T for k in range(3))
        Gp_ref = dH * dact(H64)          # Hin plays the role of the previous layer's OUTPUT
        assert _relmax(from_dev(tGp), Gp_ref) <= 2e-5
    torch.cuda.synchronize()


@pytest.mark.parametrize('cin,cout', [(16, 16), (32, 32), (16, 32), (32, 16), (64, 32)])
@pytest.mark.parametrize('family,b', [(0, 19), (0, 24), (1, 24), (1, 19), (1, 48)])
def test_occupancy_flags_are_exact(small, cin, cout, family, b):
    """Row-sparse features: the flagged kernels (skip zero neighbour rows / zero tiles) must reproduce the unflagged
    kernels bit for bit, and the flags they emit must be a superset of the non-zero rows.  family 0 = fp32 SIMT kernels
    (dense tiles vs unit kernels), family 1 = tensor-core kernels (dense slabs vs compacted row lists; b % 4 != 0 falls back
    to the unit kernels, whose results then differ from the slab kernel by fp32 rounding noise only)."""
    sg = _mods()
    from scone_gcn_b200 import _lib
    L = _lib.lib()
    cx = sg.SimplicialComplex.from_dense(small.B1, small.B2, 'scone')
    E = cx.E
    dev = torch.device('cuda')
    g = torch.Generator(device='cpu').manual_seed(cin + cout)
    keep = (torch.rand(E, b, 1, generator=g) < 0.05).float()
    H = (torch.randn(E, b, cin, generator=g) * keep).to(dev)
    G = (torch.randn(E, b, cout, generator=g) * (torch.rand(E, b, 1, generator=g) < 0.03).float()).to(dev)
    occH = (H.abs().amax(dim=2) > 0).to(torch.uint8).contiguous()
    occG = (G.abs().amax(dim=2) > 0).to(torch.uint8).contiguous()
    W = [(torch.randn(cin, cout, generator=g) * 0.3).to(dev) for _ in range(3)]
    st = torch.cuda.current_stream().cuda_stream
    outs = []
    scratch = torch.empty(L.scone_occ_scratch_bytes(cx.handle, b), dtype=torch.uint8, device=dev)
    L.scone_set_dense_kernel(family)
    for flagged in (0, 1, 2):
        out = torch.full((E, b, cout), 7.0, device=dev)
        occ_out = torch.full((E, b), 9, dtype=torch.uint8, device=dev)
        _lib.check(L.scone_layer_forward(cx.handle, 0, b, cin, cout, _lib.dptr(H), _lib.dptr(W[0]), _lib.dptr(W[1]), _lib.dptr(W[2]),
                                         _lib.dptr(out), _lib.dptr(occH) if flagged else None, _lib.dptr(occ_out),
                                         _lib.dptr(scratch) if flagged else None, st))
        ws = torch.empty(L.scone_layer_backward_workspace_bytes(cin, cout) // 4 + 16, device=dev)
        dW = torch.zeros(3, cin, cout, device=dev)
        Gp = torch.full((E, b, cin), 7.0, device=dev)
        occ_p = torch.full((E, b), 9, dtype=torch.uint8, device=dev)
        _lib.check(L.scone_layer_backward(cx.handle, 0, b, cin, cout, _lib.dptr(G), _lib.dptr(H), _lib.dptr(W[0]), _lib.dptr(W[1]),
                                          _lib.dptr(W[2]), _lib.dptr(Gp), _lib.dptr(dW), 0, _lib.dptr(ws),
                                          _lib.dptr(occG) if flagged else None, _lib.dptr(occH) if flagged == 2 else None,
                                          _lib.dptr(occ_p), _lib.dptr(scratch) if flagged else None, st))
        outs.append((out.cpu(), occ_out.cpu(), Gp.cpu(), occ_p.cpu(), dW.cpu()))
    L.scone_set_dense_kernel(_lib.DEFAULT_DENSE_KERNEL)
    same_arith = family == 0 or cin == 64 or b % (128 // cin) == 0      # else: slab (3xTF32) vs unit (fp32 SIMT) kernels
    for k in (1, 2):
        if same_arith:
            assert torch.equal(outs[0][0], outs[k][0])                                         # Hout bit-identical
        else:
            assert (outs[0][0] - outs[k][0]).abs().max() <= 2e-5
        assert torch.equal(outs[0][2], outs[k][2])                                             # Gprev bit-identical
        assert _relmax(outs[k][4].numpy(), outs[0][4].numpy()) < 1e-5                          # dW: other summation order
        assert not ((outs[k][0].abs().amax(dim=2) > 0) & ~outs[k][1].bool()).any()            # flags cover the non-zero rows
        assert not ((outs[k][2].abs().amax(dim=2) > 0) & ~outs[k][3].bool()).any()
    assert torch.equal(outs[1][4], outs[2][4])
    assert outs[0][1].min() == 1                                 # dense kernels carry no information: everything flagged
    assert 0 < outs[1][1].float().mean() < 0.9


@pytest.mark.parametrize('cin,cout,act', [(16, 16, 0), (32, 32, 0), (16, 32, 1), (32, 16, 2)])
@pytest.mark.parametrize('b', [3, 16, 40])
def test_slab_kernels_match_simt_dense_kernels(small, cin, cout, act, b):
    """The tensor-core slab kernels (3xTF32, both slab shapes) against the fp32 SIMT dense kernels on the same input:
    same gather order, product within fp32 rounding noise; ragged trajectory counts included."""
    sg = _mods()
    from scone_gcn_b200 import _lib
    L = _lib.lib()
    cx = sg.SimplicialComplex.from_dense(small.B1, small.B2, 'scone')
    E = cx.E
    dev = torch.device('cuda')
    g = torch.Generator(device='cpu').manual_seed(7 * cin + cout + b)
    H = torch.randn(E, b, cin, generator=g).to(dev)
    W = [(torch.randn(cin, cout, generator=g) * 0.3).to(dev) for _ in range(3)]
    st = torch.cuda.current_stream().cuda_stream
    outs = []
    try:
        for which in (0, 1, 2):
            L.scone_set_dense_kernel(which)
            out = torch.full((E, b, cout), 7.0, device=dev)
            _lib.check(L.scone_layer_forward(cx.handle, act, b, cin, cout, _lib.dptr(H), _lib.dptr(W[0]), _lib.dptr(W[1]),
                                             _lib.dptr(W[2]), _lib.dptr(out), None, None, None, st))
            outs.append(out.cpu().numpy())
    finally:
        L.scone_set_dense_kernel(_lib.DEFAULT_DENSE_KERNEL)
    scale = max(1.0, np.abs(outs[0]).max())
    for k in (1, 2):
        assert np.abs(outs[k] - outs[0]).max() <= 2e-5 * scale, (k, np.abs(outs[k] - outs[0]).max())


@pytest.mark.parametrize('mb', [32, 7])
def test_unit_kernel_pipeline_is_bit_identical_run_to_run(small, mb):
    """Pipeline 0 (unit kernels over byte flags): two passes of forward + loss/gradient give the same log-probs and gradients bit
    for bit (rows outside the support are never written, so the second pass runs over the tensors the first left behind), and the
    log-probs match the reference fixture."""
    sg = _mods()
    fx = load('model_small_scone_h16.npz')
    cx = sg.SimplicialComplex.from_dense(small.B1, small.B2, 'scone')
    ptr, fe, fv = sg.flows_to_csr(small.flows)
    net = sg.SconeModel(cx, [16, 16, 16], micro_batch=mb)
    net.set_pipeline(0)
    net.set_weights(weights_of(fx, 'w_big'))
    res = []
    for _ in range(2):
        lp = net.forward(ptr, fe, fv, small.last_nodes)
        buf = net.loss_grad(ptr, fe, fv, small.last_nodes, small.raw['targets_argmax'], np.ones(small.n_traj, np.float32))
        res.append((lp, buf))
    assert np.array_equal(res[0][0], res[1][0]) and np.array_equal(res[0][1], res[1][1])
    assert np.abs(res[0][0] - fx['big_logprobs'][:, :, 0]).max() < 1e-5


@pytest.mark.parametrize('model,hidden,mb', [('scone', [16, 16, 16], 32), ('scone', [32, 32, 32], 7), ('ebli', [16, 32, 16], 64),
                                             ('scone', [32], 16), ('scone', [16, 32], 5), ('scone', [16, 16, 16, 16], 13),
                                             ('ebli', [32, 32, 32, 32], 40)])
def test_row_list_pipeline_matches_unit_kernel_pipeline(small, model, hidden, mb):
    """Model level: the bitmap-native row-list pipelines (tensor-core kernels; 3 = compact tensors over the readout cone,
    2 = compact tensors over the whole support, 1 = dense tensors) against the unit-kernel pipeline (0: fp32 SIMT, byte flags):
    log-probs within 1e-5, gradients within 1e-4 of the largest entry; run-to-run bit-exact; interleaving the pipelines on one
    model (X must be re-cleaned) changes nothing; and pruning to the cone changes no bit of the log-probs (gradients: 1e-5)."""
    sg = _mods()
    L = sg.lib()
    cx = sg.SimplicialComplex.from_dense(small.B1, small.B2, model)
    ptr, fe, fv = sg.flows_to_csr(small.flows)
    net = sg.SconeModel(cx, hidden, micro_batch=mb)
    assert L.scone_model_get_pipeline(net.handle) in (3, 4)        # default: fused (uniform widths, <= 3 layers) or cone row lists
    rs = np.random.RandomState(len(hidden) * 10 + mb)
    net.set_weights([0.1 * rs.randn(*s_) for s_ in net.shapes])
    mask = (rs.rand(small.n_traj) < 0.7).astype(np.float32)
    out = {}
    for which in (3, 2, 1, 0, 3, 2, 1):
        _lib_check = __import__('scone_gcn_b200')._lib.check
        _lib_check(L.scone_model_set_pipeline(net.handle, which), 'set_pipeline')
        lp = net.forward(ptr, fe, fv, small.last_nodes)
        buf = net.loss_grad(ptr, fe, fv, small.last_nodes, small.raw['targets_argmax'], mask)
        if which in out:
            assert np.array_equal(out[which][0], lp) and np.array_equal(out[which][1], buf)
        out[which] = (lp, buf)
    assert np.array_equal(out[2][0], out[1][0])                    # compact vs dense addressing: same arithmetic per row
    # cone pruning: the log-probs do not change by a bit; the weight gradients lose only exact-zero terms (their sums are grouped
    # differently: fp32 summation noise)
    assert np.array_equal(out[3][0], out[2][0])
    n = net.n_params
    assert np.array_equal(out[3][1][n:], out[2][1][n:])
    off = 0
    for shp in net.shapes:
        k = shp[0] * shp[1]
        assert np.abs(out[3][1][off:off + k] - out[2][1][off:off + k]).max() <= 1e-5 * max(np.abs(out[2][1][off:off + k]).max(), 1e-30), shp
        off += k
    for which in (1, 2, 3):
        assert np.abs(out[which][0] - out[0][0]).max() <= 1e-5 * max(1.0, np.abs(out[0][0]).max())
        assert out[which][1][n + 1] == out[0][1][n + 1] == mask.sum()
        assert abs(out[which][1][n] - out[0][1][n]) <= 1e-5 * max(1.0, abs(out[0][1][n]))
        off = 0
        for shp in net.shapes:
            k = shp[0] * shp[1]
            a, r = out[which][1][off:off + k], out[0][1][off:off + k]
            assert np.abs(a - r).max() <= 1e-4 * max(np.abs(r).max(), 1e-30), (which, shp)
            off += k


def test_training_matches_oracle_end_to_end(small):
    """k Adam steps from the reference init / batch stream: same weights (1e-4) and identical accuracy."""
    sg = _mods()
    fx = load('model_small_scone_h16.npz')
    from scone_gcn_b200.scone_trajectory_model import Scone_GCN
    from scone_gcn_b200 import trajectory_experiments as te
    np.random.seed(1030)
    cx = sg.SimplicialComplex.from_dense(small.B1, small.B2, 'scone')
    shifts = te.shift_handles(cx)
    inputs = [te.Bconds(cx), small.last_nodes, small.flows]
    net = Scone_GCN(int(fx['epochs']), float(fx['lr']), int(fx['batch_size']), float(fx['wd']), verbose=False)
    in_axes = (None, None, None, None, 0, 0)
    net.setup(te.scone_func, [(3, 16)] * 3, shifts, inputs, small.targets, in_axes, small.train_mask)
    for a, r in zip(net.weights, weights_of(fx, 'w_init')):
        assert np.array_equal(np.asarray(a), r)
    res = net.train(inputs, small.targets, small.train_mask, small.test_mask, fx['n_nbrs'])
    ref = fx['train_result']
    assert res[0] == pytest.approx(ref[0], rel=1e-4) and res[2] == pytest.approx(ref[2], rel=1e-4)
    assert res[1] == pytest.approx(ref[1], abs=1e-7) and res[3] == pytest.approx(ref[3], abs=1e-7)
    for i, w in enumerate(net.weights):
        assert _relmax(np.asarray(w), fx['w_trained_%d' % i]) <= 2e-3, i      # 9 Adam steps amplify fp32 noise


def test_default_complex_training_matches_oracle():
    """cfg1: 3 epochs (24 Adam steps) of the default run from the reference init and batch stream; the oracle runs the
    reference formulation (dense E x E, forward over all 1000 trajectories, autograd) on the CPU beside it."""
    sg = _mods()
    from scone_gcn_b200.scone_trajectory_model import Scone_GCN
    from scone_gcn_b200 import trajectory_experiments as te
    ds = Dataset('dataset_default.npz')
    fx = load('model_default_scone_h16.npz')
    epochs, bs, lr, wd = 3, 100, 1e-3, 5e-5
    # oracle
    orc = so.DenseOracle('scone', so.shift_matrices(ds.B1, ds.B2, 'scone'), ds.B1, ds.last_nodes, ds.flows, ds.targets)
    rng = np.random.RandomState(1030)
    W0 = so.generate_weights(rng, 1, [(3, 16)] * 3, 1, 'scone')
    Wo, res_o = so.train(orc, rng, W0, ds.train_mask, ds.test_mask, epochs, bs, lr, wd)
    # CUDA path through the reference API
    np.random.seed(1030)
    cx = sg.SimplicialComplex.from_simplices(ds.N, ds.edges, ds.faces, 'scone')
    inputs = [te.Bconds(cx), ds.last_nodes, ds.flows]
    net = Scone_GCN(epochs, lr, bs, wd, verbose=False)
    net.setup(te.scone_func, [(3, 16)] * 3, te.shift_handles(cx), inputs, ds.targets, None, ds.train_mask)
    res = net.train(inputs, ds.targets, ds.train_mask, ds.test_mask, fx['n_nbrs'])
    assert res[0] == pytest.approx(res_o[0], rel=1e-4) and res[2] == pytest.approx(res_o[2], rel=1e-4)
    assert res[1] == pytest.approx(res_o[1], abs=1e-9) and res[3] == pytest.approx(res_o[3], abs=1e-9)   # identical accuracy
    for a, b in zip(net.weights, Wo):
        assert _relmax(np.asarray(a), b) <= 5e-3

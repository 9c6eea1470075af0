"""The tcgen05 / TMEM dense layer kernel (csrc/scone_umma.cu, scone_set_dense_kernel(3)) through the C ABI against the fp32 SIMT dense
kernel on the same input: same gather order, 3xTF32 product within fp32 rounding noise; complexes whose edge count is not a
multiple of the 8-edge tile, several trajectory-slab counts, all three activations."""
import numpy as np
import pytest
import torch

from golden_util import Dataset

pytestmark = pytest.mark.gpu


def _run(cx, act, b, H, W, which):
    from scone_gcn_b200 import _lib
    L = _lib.lib()
    st = torch.cuda.current_stream().cuda_stream
    L.scone_set_dense_kernel(which)
    try:
        out = torch.full((cx.E, b, 32), 7.0, device=H.device)
        _lib.check(L.scone_layer_forward(cx.handle, act, b, 32, 32, _lib.dptr(H), _lib.dptr(W[0]), _lib.dptr(W[1]), _lib.dptr(W[2]),
                                         _lib.dptr(out), None, None, None, st))
        if which == 3:
            _lib.check(L.scone_umma_status(st), 'scone_umma_status')
        return out.cpu().numpy()
    finally:
        L.scone_set_dense_kernel(_lib.DEFAULT_DENSE_KERNEL)


@pytest.mark.parametrize('act', [0, 1, 2])
@pytest.mark.parametrize('b', [16, 48, 64])
def test_umma_forward_matches_simt_dense_kernel(act, b):
    import scone_gcn_b200 as sg
    ds = Dataset('dataset_small.npz')
    cx = sg.SimplicialComplex.from_dense(ds.B1, ds.B2, 'scone')
    dev = torch.device('cuda')
    g = torch.Generator(device='cpu').manual_seed(100 + 7 * act + b)
    H = torch.randn(cx.E, b, 32, generator=g).to(dev)
    W = [(torch.randn(32, 32, generator=g) * 0.3).to(dev) for _ in range(3)]
    ref = _run(cx, act, b, H, W, 0)
    got = _run(cx, act, b, H, W, 3)
    assert np.abs(got - ref).max() <= 2e-5 * max(1.0, np.abs(ref).max()), np.abs(got - ref).max()


def test_umma_forward_on_a_larger_sparse_complex_many_tiles_per_cta():
    """~9000 edges x 64 trajectories: hundreds of tiles, both warp groups of every CTA cycle through many mbarrier phases."""
    import scone_gcn_b200 as sg
    from scone_gcn_b200 import synthetic_data_gen as sdg
    sp = sdg.generate_sparse_dataset(3000, 8, seed=5, n_waypoints=8)
    cx = sg.SimplicialComplex.from_simplices(int(sp.n_nodes), sp.edges, sp.faces, 'scone')
    dev = torch.device('cuda')
    g = torch.Generator(device='cpu').manual_seed(3)
    b = 64
    H = torch.randn(cx.E, b, 32, generator=g).to(dev)
    W = [(torch.randn(32, 32, generator=g) * 0.2).to(dev) for _ in range(3)]
    ref = _run(cx, 0, b, H, W, 1)                          # slab kernel (mma.sync 3xTF32): same gather, same split
    got = _run(cx, 0, b, H, W, 3)
    assert np.abs(got - ref).max() <= 1e-5 * max(1.0, np.abs(ref).max()), np.abs(got - ref).max()
    got2 = _run(cx, 0, b, H, W, 3)
    assert np.array_equal(got, got2)                       # run-to-run bit-exact


def _run_bwd(cx, act, b, G, H, W, which, with_gprev=True):
    from scone_gcn_b200 import _lib
    L = _lib.lib()
    st = torch.cuda.current_stream().cuda_stream
    L.scone_set_dense_kernel(which)
    try:
        Gp = torch.full((cx.E, b, 32), 7.0, device=H.device) if with_gprev else None
        dW = torch.full((3, 32, 32), 0.5, device=H.device)
        ws = torch.empty(L.scone_layer_backward_workspace_bytes(32, 32) // 4 + 16, device=H.device)
        _lib.check(L.scone_layer_backward(cx.handle, act, b, 32, 32, _lib.dptr(G), _lib.dptr(H), _lib.dptr(W[0]), _lib.dptr(W[1]),
                                          _lib.dptr(W[2]), _lib.dptr(Gp) if with_gprev else None, _lib.dptr(dW), 1, _lib.dptr(ws),
                                          None, None, None, None, st))
        if which == 3:
            _lib.check(L.scone_umma_status(st), 'scone_umma_status')
        return (Gp.cpu().numpy() if with_gprev else None), dW.cpu().numpy() - 0.5
    finally:
        L.scone_set_dense_kernel(_lib.DEFAULT_DENSE_KERNEL)


@pytest.mark.parametrize('act', [0, 1, 2])
@pytest.mark.parametrize('b', [16, 48])
def test_umma_backward_matches_float64(act, b):
    """tcgen05 backward (weight gradient accumulated in TMEM over K = rows, operands in shared memory; row product on mma.sync)
    against a float64 restatement of what jax.grad derives (scone_trajectory_model.py:307); accumulate = 1 adds onto dW."""
    import scone_gcn_b200 as sg
    ds = Dataset('dataset_small.npz')
    cx = sg.SimplicialComplex.from_dense(ds.B1, ds.B2, 'scone')
    dev = torch.device('cuda')
    g = torch.Generator(device='cpu').manual_seed(200 + 7 * act + b)
    Hc = torch.tanh(torch.randn(cx.E, b, 32, generator=g))
    Gc = torch.randn(cx.E, b, 32, generator=g)
    Wc = [torch.randn(32, 32, generator=g) * 0.3 for _ in range(3)]
    rank = torch.from_numpy(cx.edge_rank.astype(np.int64))          # device tensors use the internal edge order
    Hd = torch.empty_like(Hc)
    Gd = torch.empty_like(Gc)
    Hd[rank] = Hc
    Gd[rank] = Gc
    Gp, dW = _run_bwd(cx, act, b, Gd.to(dev), Hd.to(dev), [w.to(dev) for w in Wc], 3)
    S = [cx.shift_dense(0), cx.shift_dense(1)]
    G64, H64 = Gc.numpy().astype(np.float64), Hc.numpy().astype(np.float64)
    A = [G64, np.einsum('ef,fbc->ebc', S[0], G64), np.einsum('ef,fbc->ebc', S[1], G64)]
    dW_ref = np.stack([np.einsum('ebi,ebo->io', H64, A[k]) for k in range(3)])
    dH = sum(A[k] @ Wc[k].numpy().astype(np.float64).T for k in range(3))
    dact = (1 - H64 * H64) if act == 0 else (np.where(H64 >= 0, 1.0, 0.01) if act == 1 else (H64 > 0).astype(np.float64))
    Gp_ref = dH * dact
    assert np.abs(dW - dW_ref).max() <= 2e-5 * np.abs(dW_ref).max(), np.abs(dW - dW_ref).max() / np.abs(dW_ref).max()
    assert np.abs(Gp[rank.numpy()] - Gp_ref).max() <= 2e-5 * max(1.0, np.abs(Gp_ref).max())
    _, dW_only = _run_bwd(cx, act, b, Gd.to(dev), Hd.to(dev), [w.to(dev) for w in Wc], 3, with_gprev=False)
    assert np.array_equal(dW_only, dW)                     # first-use variant (no Gprev): the same TMEM accumulation


def test_umma_backward_many_slabs_per_warp_and_in_place():
    """~9000 edges x 64 trajectories: every warp runs through many mbarrier phases; against the fp32 SIMT tile kernel; run-to-run
    bit-exact; Gprev may alias Hin (bench.py's dense figure calls it that way)."""
    import scone_gcn_b200 as sg
    from scone_gcn_b200 import synthetic_data_gen as sdg
    sp = sdg.generate_sparse_dataset(3000, 8, seed=5, n_waypoints=8)
    cx = sg.SimplicialComplex.from_simplices(int(sp.n_nodes), sp.edges, sp.faces, 'scone')
    dev = torch.device('cuda')
    g = torch.Generator(device='cpu').manual_seed(4)
    b = 64
    H = torch.tanh(torch.randn(cx.E, b, 32, generator=g)).to(dev)
    G = torch.randn(cx.E, b, 32, generator=g).to(dev)
    W = [(torch.randn(32, 32, generator=g) * 0.2).to(dev) for _ in range(3)]
    Gp0, dW0 = _run_bwd(cx, 0, b, G, H, W, 0)
    Gp3, dW3 = _run_bwd(cx, 0, b, G, H, W, 3)
    assert np.abs(Gp3 - Gp0).max() <= 1e-5 * max(1.0, np.abs(Gp0).max())
    assert np.abs(dW3 - dW0).max() <= 2e-5 * np.abs(dW0).max()
    Gp3b, dW3b = _run_bwd(cx, 0, b, G, H, W, 3)
    assert np.array_equal(Gp3, Gp3b) and np.array_equal(dW3, dW3b)
    from scone_gcn_b200 import _lib
    L = _lib.lib()
    st = torch.cuda.current_stream().cuda_stream
    Hc = H.clone()
    dW = torch.zeros(3, 32, 32, device=dev)
    ws = torch.empty(L.scone_layer_backward_workspace_bytes(32, 32) // 4 + 16, device=dev)
    L.scone_set_dense_kernel(3)
    try:
        _lib.check(L.scone_layer_backward(cx.handle, 0, b, 32, 32, _lib.dptr(G), _lib.dptr(Hc), _lib.dptr(W[0]), _lib.dptr(W[1]),
                                          _lib.dptr(W[2]), _lib.dptr(Hc), _lib.dptr(dW), 0, _lib.dptr(ws), None, None, None, None, st))
        _lib.check(L.scone_umma_status(st), 'scone_umma_status')
    finally:
        L.scone_set_dense_kernel(_lib.DEFAULT_DENSE_KERNEL)
    assert np.array_equal(Hc.cpu().numpy(), Gp3) and np.array_equal(dW.cpu().numpy(), dW3)

"""Vector-Jacobian product of the log-probs (scone_model_vjp_*, scone_bunch_vjp_host, scone_gcn_b200.torch_ops): the readout's dlogit
seed generalised from a one-hot target to any upstream gradient cot[t][j] = dL/dlogprob[t][j].

  - with cot = -mask * onehot(target) and count_add = sum(mask) (masks in {0, 1}) the buffer is bit for bit loss_grad's, on every
    pipeline and on the bunch model;
  - dense random cotangents (padded slots and all-zero rows included) against torch.autograd.grad(lp, W, cot) of the float64 oracle,
    at every layer-width path, the BIG launch, high degrees and on the bunch model, whose padded slots read node N - 1;
  - the torch autograd op under a nonlinear loss; Scone_GCN.train on soft targets against a float64 restatement of the reference's
    grad(-sum(preds * y) / sum(mask) + ridge) and Adam.
Tolerances are the suite's: weight gradients 1e-4 of their largest entry (with the noise floor of test_gpu_tiny_complexes.py), the
nll_sum slot 1e-5 relative to the sum of |cot * logprob|, count exact."""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from golden_util import Dataset
from oracle import scone_oracle as so
from scone_gcn_b200.bunch_model_matrices import compute_shift_matrices
from test_gpu_bunch import SparseBunchRef, calibrated_weights, dataset_problem
from test_gpu_high_degree import fused_net, problem, scaled_weights

pytestmark = pytest.mark.gpu


def onehot_cot(tgt, mask, D):
    cot = np.zeros((len(tgt), D), np.float32)
    cot[np.arange(len(tgt)), tgt] = 1.0
    return -mask[:, None].astype(np.float32) * cot


def random_cot(rs, B, D, zero_rows=(1, 4)):
    """Dense cotangents, mostly positive (the log-probs are <= 0, so the nll_sum slot does not cancel), with all-zero rows (the rows
    a mask drops)."""
    cot = rs.uniform(-0.25, 1.0, size=(B, D)).astype(np.float32)
    cot[list(zero_rows)] = 0.0
    return cot


def oracle_vjp(forward, W, cot):
    """(logprobs [B, D], sum cot * lp, [d/dW sum cot * lp]) in float64; forward(W list of tensors) -> [B, D]."""
    W = [torch.as_tensor(np.asarray(w, np.float64)).requires_grad_(True) for w in W]
    lp = forward(W)
    c = torch.as_tensor(np.asarray(cot, np.float64))
    ell = (lp * c).sum()
    g = torch.autograd.grad(ell, W, allow_unused=True)      # (bunch: the last layer's edge / triangle weights never reach the readout)
    return lp.detach().numpy(), float(ell.detach()), [np.zeros(w.shape) if x is None else x.numpy() for w, x in zip(W, g)]


def check_buffer(buf, n_params, unflatten, lp_ref, ell_ref, g_ref, cot, count_add, what):
    assert buf[n_params + 1] == np.float32(count_add), what
    bound = np.abs(np.asarray(cot, np.float64) * lp_ref).sum()
    assert abs(buf[n_params] - ell_ref) <= 1e-5 * bound, (what, 'nll_sum', buf[n_params], ell_ref)
    grads = unflatten(buf[:n_params])
    gmax = max(float(np.abs(r).max()) for r in g_ref)
    for i, (a, r) in enumerate(zip(grads, g_ref)):
        assert np.abs(a - r).max() <= 1e-4 * max(float(np.abs(r).max()), 1e-3 * gmax), (what, 'grad', i, np.abs(a - r).max(), np.abs(r).max())


def scone_setup(model, hidden, mb, scale, seed=0):
    import scone_gcn_b200 as sg
    ds = Dataset('dataset_small.npz')
    cx = sg.SimplicialComplex.from_dense(ds.B1, ds.B2, model)
    net = sg.SconeModel(cx, hidden, micro_batch=mb)
    rs = np.random.RandomState(seed)
    W = [(scale * rs.randn(*s)).astype(np.float32) for s in net.shapes]
    net.set_weights(W)
    return ds, cx, net, W


# ---- 1. one-hot cotangents: bit for bit loss_grad ------------------------------------------------------------------------------------
@pytest.mark.parametrize('variant', ['4-table', '4-hash', '4-planned', '4-host-overlap', 3, 2, 1, 0])
def test_onehot_cotangent_gives_the_loss_grad_buffer_bit_for_bit(variant, monkeypatch):
    import scone_gcn_b200 as sg
    ds = Dataset('dataset_default.npz' if variant == '4-host-overlap' else 'dataset_small.npz')
    if variant == '4-hash':
        monkeypatch.setenv('SCONE_FUSED_TABLE', '0')                # read when a model is created
    cx = sg.SimplicialComplex.from_dense(ds.B1, ds.B2, 'scone')
    mb = 1024 if variant == '4-host-overlap' else 16               # (60 trajectories: four micro-batches, the last one ragged)
    net = sg.SconeModel(cx, [16, 16, 16], micro_batch=mb)
    if isinstance(variant, int):
        net.set_pipeline(variant)
    assert net.pipeline == (variant if isinstance(variant, int) else 4)
    if variant == '4-hash':
        assert net.fused_info()['table_plan_mb'] == 0
    rs = np.random.RandomState(5)
    net.set_weights([0.2 * rs.randn(*s) for s in net.shapes])
    tgt = ds.raw['targets_argmax'].astype(np.int32)
    mask = ds.train_mask.astype(np.float32)
    ptr, fe, fv = sg.flows_to_csr(ds.flows)
    last = ds.last_nodes
    if variant == '4-planned':
        assert net.plan(ptr, fe, fv, last)
        rows = rs.permutation(ds.n_traj)[:41]
        tgt, mask = tgt[rows], mask[rows]
        ref = net.loss_grad_planned(rows, tgt, mask)
        got = net.vjp_planned(rows, onehot_cot(tgt, mask, cx.D), mask.sum())
    else:
        ref = net.loss_grad(ptr, fe, fv, last, tgt, mask)
        got = net.vjp(ptr, fe, fv, last, onehot_cot(tgt, mask, cx.D), mask.sum())
    assert (ref[:-2] != 0).any() and ref[-1] == mask.sum() and (mask == 0).any()
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))


def test_onehot_cotangent_gives_the_bunch_loss_grad_buffer_bit_for_bit():
    p = dataset_problem('small')
    ref = SparseBunchRef(p.shifts, p.nbrhoods)
    W = calibrated_weights(ref, [8, 8], p.flows, p.last_nodes, seed=2)
    net = p.model([8, 8], micro_batch=16)
    net.set_weights(W)
    ptr, fe, fv = p.csr()
    a = net.loss_grad(ptr, fe, fv, p.last_nodes, p.tgt, p.mask)
    b = net.vjp(ptr, fe, fv, p.last_nodes, onehot_cot(p.tgt, p.mask, p.D), p.mask.sum())
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32))


# ---- 2. / 5. random cotangents against the float64 oracle, determinism ------------------------------------------------------------
CASES = [('scone', [16, 16, 16], 4, False, 0.1), ('scone', [16, 16, 16], 4, True, 0.1), ('scone', [32, 32, 32], 4, False, 0.1),
         ('scone', [32, 32, 32], 4, True, 0.1), ('ebli', [32, 32, 32], 4, False, 0.03), ('scone', [16, 32, 16], 3, False, 0.1),
         ('scone', [8, 8, 8], 0, False, 0.2), ('scone', [64], 0, False, 0.2), ('scone', [16, 16, 16, 16], 3, False, 0.15)]


@pytest.mark.parametrize('model,hidden,pipeline,planned,scale', CASES,
                         ids=['%s-%s-p%d%s' % (c[0], 'x'.join(map(str, c[1])), c[2], '-planned' if c[3] else '') for c in CASES])
def test_random_cotangents_match_the_float64_oracle(model, hidden, pipeline, planned, scale):
    import scone_gcn_b200 as sg
    ds, cx, net, W = scone_setup(model, hidden, 16, scale)
    assert net.pipeline == pipeline
    rs = np.random.RandomState(len(hidden) + hidden[0])
    B = ds.n_traj
    cot = random_cot(rs, B, cx.D)
    orc = so.DenseOracle(model, so.shift_matrices(ds.B1, ds.B2, model), ds.B1, ds.last_nodes, ds.flows, ds.targets, dtype=torch.float64)
    if planned:
        ptr, fe, fv = sg.flows_to_csr(ds.flows)
        assert net.plan(ptr, fe, fv, ds.last_nodes)
        rows = rs.permutation(B)[:45]
        lp_ref, ell, g_ref = oracle_vjp(lambda Wt: orc.forward(Wt, torch.as_tensor(rows))[:, :, 0], W, cot[rows])
        bufs = [net.vjp_planned(rows, cot[rows], 3.0) for _ in range(2)]
        check_buffer(bufs[0], net.n_params, net.unflatten, lp_ref, ell, g_ref, cot[rows], 3.0, 'planned')
    else:
        ptr, fe, fv = sg.flows_to_csr(ds.flows)
        lp_ref, ell, g_ref = oracle_vjp(lambda Wt: orc.forward(Wt)[:, :, 0], W, cot)
        bufs = [net.vjp(ptr, fe, fv, ds.last_nodes, cot, 7.0) for _ in range(2)]
        check_buffer(bufs[0], net.n_params, net.unflatten, lp_ref, ell, g_ref, cot, 7.0, 'unplanned')
        if model == 'ebli':                                        # the BIG launch (rows beyond the shared-memory store) took part
            info = net.fused_info()
            whole = sg.SconeModel(cx, hidden, micro_batch=B)
            whole.set_weights(W)
            whole.forward(ptr, fe, fv, ds.last_nodes)
            assert max(int(whole.fused_header(t)[1:4].sum()) for t in range(B)) > info['cap_rows']
    assert np.array_equal(bufs[0].view(np.uint32), bufs[1].view(np.uint32))      # deterministic


# ---- 3. high degree: small and BIG launch, cotangent mass on padded slots -----------------------------------------------------------
@pytest.mark.parametrize('name', ['wheel_72', 'hubs_8x120'])
def test_high_degree_cotangents_with_padded_mass_match_the_oracle(name, monkeypatch):
    hidden = [32, 32, 32]
    p = problem(name, 'scone', 3, seed=29)
    S = [sp.csr_matrix(m) for m in so.shift_matrices(p['B1'], p['B2'], 'scone')]
    W, peaks = scaled_weights('scone', p['B1'], S, p['flows'][:, :, 0], p['last'], hidden, np.random.RandomState(11))
    assert all(1.0 <= q <= 4.0 for q in peaks), peaks
    B, D = len(p['last']), p['cx'].D
    rs = np.random.RandomState(3)
    cot = random_cot(rs, B, D)
    padded = np.arange(D)[None, :] >= p['n_nbrs'][:, None]
    assert padded.any()
    cot[padded] *= 4.0                                             # most of the mass on slots with no real neighbour
    net = fused_net(monkeypatch, p, hidden, W, 'table', B)
    ptr, fe, fv = p['csr']
    net.forward(ptr, fe, fv, p['last'])
    rows = np.array([int(net.fused_header(t)[1:4].sum()) for t in range(B)])
    cap = net.fused_info()['cap_rows']
    assert (rows > cap).any() and (rows <= cap).any()              # both launches of the compute kernel
    orc = so.DenseOracle('scone', so.shift_matrices(p['B1'], p['B2'], 'scone'), p['B1'], p['last'], p['flows'], p['targets'],
                         dtype=torch.float64)
    lp_ref, ell, g_ref = oracle_vjp(lambda Wt: orc.forward(Wt)[:, :, 0], W, cot)
    buf = net.vjp(ptr, fe, fv, p['last'], cot, 5.0)
    check_buffer(buf, net.n_params, net.unflatten, lp_ref, ell, g_ref, cot, 5.0, name)


# ---- 4. bunch ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('hidden', [[16, 16, 16], [8, 12, 16]], ids=lambda h: 'x'.join(map(str, h)))
@pytest.mark.parametrize('where', ['dense', 'padded-only'])
def test_bunch_cotangents_match_the_float64_reference(hidden, where):
    p = dataset_problem('small')
    ref = SparseBunchRef(p.shifts, p.nbrhoods)
    W = calibrated_weights(ref, hidden, p.flows, p.last_nodes, seed=4)
    rs = np.random.RandomState(len(hidden) + hidden[1])
    cot = random_cot(rs, p.B, p.D)
    padded = p.nbrhoods[p.last_nodes] < 0
    assert padded.any()
    if where == 'padded-only':                                     # only slots that read node N - 1 carry a cotangent
        cot[~padded] = 0.0
    net = p.model(hidden, micro_batch=16)
    net.set_weights(W)
    ptr, fe, fv = p.csr()
    lp_ref, ell, g_ref = oracle_vjp(lambda Wt: ref.forward(Wt, p.flows, p.last_nodes), W, cot)
    bufs = [net.vjp(ptr, fe, fv, p.last_nodes, cot, 2.0) for _ in range(2)]
    check_buffer(bufs[0], net.n_params, net.unflatten, lp_ref, ell, g_ref, cot, 2.0, where)
    assert np.array_equal(bufs[0].view(np.uint32), bufs[1].view(np.uint32))


# ---- 6. the torch autograd op -------------------------------------------------------------------------------------------------------
def soft_loss(lp, q, padded):
    """KL(q || p) plus a nonlinear term on the padded slots."""
    return (q * (torch.log(q) - lp)).sum() + 0.5 * (torch.exp(lp) * padded).sum() ** 2


def test_torch_op_gradient_of_a_nonlinear_loss_matches_the_oracle():
    import scone_gcn_b200 as sg
    from scone_gcn_b200 import torch_ops
    ds, cx, net, W = scone_setup('scone', [16, 16, 16], 32, 0.2)
    assert net.pipeline == 4
    dev = torch.device('cuda')
    ptr, fe, fv = sg.flows_to_csr(ds.flows)
    args = [torch.as_tensor(a, device=dev) for a in (ptr, fe, fv, ds.last_nodes.astype(np.int32))]
    rs = np.random.RandomState(9)
    q64 = rs.dirichlet(np.ones(cx.D), size=ds.n_traj)
    nb, _, _ = so.neighbourhood_tables(ds.B1, ds.last_nodes)
    pad64 = (nb[ds.last_nodes] < 0).astype(np.float64)
    assert pad64.any()
    w = torch.as_tensor(net.flatten(W), device=dev).requires_grad_(True)
    lp = torch_ops.logprobs(net, w, *args)
    q, pad = torch.as_tensor(q64, dtype=torch.float32, device=dev), torch.as_tensor(pad64, dtype=torch.float32, device=dev)
    loss = soft_loss(lp, q, pad)
    net.set_weights([np.zeros(s, np.float32) for s in net.shapes])        # the model's weights change between forward and backward
    g, = torch.autograd.grad(loss, w)
    orc = so.DenseOracle('scone', so.shift_matrices(ds.B1, ds.B2, 'scone'), ds.B1, ds.last_nodes, ds.flows, ds.targets, dtype=torch.float64)
    Wt = [torch.as_tensor(np.asarray(x, np.float64)).requires_grad_(True) for x in W]
    lp64 = orc.forward(Wt)[:, :, 0]
    assert np.abs(lp.detach().cpu().numpy() - lp64.detach().numpy()).max() <= 1e-5 * max(1.0, float(lp64.detach().abs().max()))
    g_ref = torch.autograd.grad(soft_loss(lp64, torch.as_tensor(q64), torch.as_tensor(pad64)), Wt)
    gmax = max(float(r.abs().max()) for r in g_ref)
    for i, (a, r) in enumerate(zip(net.unflatten(g.cpu().numpy()), g_ref)):
        r = r.numpy()
        assert np.abs(a - r).max() <= 1e-4 * max(float(np.abs(r).max()), 1e-3 * gmax), (i, np.abs(a - r).max(), np.abs(r).max())
    # the same gradient once more after yet other weights were written: bit for bit
    net.set_weights([np.ones(s, np.float32) for s in net.shapes])
    g2, = torch.autograd.grad(soft_loss(torch_ops.logprobs(net, w, *args), q, pad), w)
    assert torch.equal(g, g2)


def test_torch_op_on_an_empty_batch():
    from scone_gcn_b200 import torch_ops
    ds, cx, net, W = scone_setup('scone', [16, 16, 16], 32, 0.2)
    dev = torch.device('cuda')
    w = torch.as_tensor(net.flatten(W), device=dev).requires_grad_(True)
    i32 = lambda n: torch.zeros(n, dtype=torch.int32, device=dev)
    lp = torch_ops.logprobs(net, w, i32(1), i32(0), torch.zeros(0, device=dev), i32(0))
    assert lp.shape == (0, cx.D)
    g, = torch.autograd.grad(lp.sum(), w)
    assert g.shape == (net.n_params,) and not g.any()


# ---- 7. soft-target training through Scone_GCN.train --------------------------------------------------------------------------------
def restated_training(orc, W0, y, batch_masks, lr, wd):
    """Float64 restatement of the reference's steps: grad(-sum(preds * y) / sum(mask) + ridge) (scone_trajectory_model.py:42-56,307)
    and the Adam formula of oracle.adam_update."""
    orc.y = torch.as_tensor(np.asarray(y, np.float64)).reshape(orc.y.shape)
    state = [(np.asarray(w, np.float64), np.zeros(np.shape(w)), np.zeros(np.shape(w))) for w in W0]
    for i, bm in enumerate(batch_masks):
        _, g = orc.loss_and_grads([s[0] for s in state], bm.astype(np.int64), wd)
        state = so.adam_update(i, g, state, lr, dtype=np.float64)
    return [s[0] for s in state]


@pytest.mark.parametrize('model', ['scone', 'bunch'])
def test_soft_target_training_follows_the_reference_gradient(model):
    import scone_gcn_b200 as sg
    from scone_gcn_b200.bunch import CsrOperator
    from scone_gcn_b200.scone_trajectory_model import Scone_GCN
    from scone_gcn_b200 import trajectory_experiments as te
    ds = Dataset('dataset_small.npz')
    rs = np.random.RandomState(17)
    y = 0.5 * ds.targets + 0.5 * rs.dirichlet(np.ones(ds.D), size=ds.n_traj)[:, :, None]      # label smoothing toward a random q
    epochs, bs, lr, wd = 1, 16, 1e-2, 5e-5
    np.random.seed(1030)
    net = Scone_GCN(epochs, lr, bs, wd, verbose=False)
    if model == 'scone':
        cx = sg.SimplicialComplex.from_dense(ds.B1, ds.B2, 'scone')
        inputs = [te.Bconds(cx), ds.last_nodes, ds.flows]
        net.setup(te.scone_func, [(3, 16)] * 3, te.shift_handles(cx), inputs, y, None, ds.train_mask)
        shifts = so.shift_matrices(ds.B1, ds.B2, 'scone')
    else:
        shifts = compute_shift_matrices(ds.B1, ds.B2)
        inputs = [so.neighbourhood_tables(ds.B1, ds.last_nodes)[0], ds.last_nodes, ds.flows]
        net.setup(te.bunch_func, [(7, 8)] * 3, [CsrOperator(M) for M in shifts], inputs, y, None, ds.train_mask, model_type='bunch')
        shifts = [M.toarray() for M in shifts]
    W0 = [np.asarray(w, np.float32) for w in net.weights]
    rng_state = np.random.get_state()
    net.train(inputs, y, ds.train_mask, ds.test_mask, so.neighbourhood_tables(ds.B1, ds.last_nodes)[1])
    if model == 'scone':
        assert net._net.planned == ds.n_traj                       # the planned-set path (vjp_planned)
    # the batch masks train() drew (scone_trajectory_model.py:318-322)
    np.random.set_state(rng_state)
    n_batches = int(ds.train_mask.sum()) // bs
    masks = []
    for _ in range(epochs * n_batches):
        bm = np.array([1] * bs + [0] * (ds.n_traj - bs))
        np.random.shuffle(bm)
        masks.append(np.logical_and(bm, ds.train_mask).astype(np.float64))
    orc = so.DenseOracle(model, shifts, ds.B1, ds.last_nodes, ds.flows, y, dtype=torch.float64)
    W_ref = restated_training(orc, W0, y, masks, lr, wd)
    W_hard = restated_training(orc, W0, ds.targets, masks, lr, wd)         # what training on argmax(y) would give
    got = [np.asarray(w, np.float64) for w in net.weights]
    err = max(float(np.abs(a - r).max()) for a, r in zip(got, W_ref))
    apart = max(float(np.abs(a - r).max()) for a, r in zip(W_hard, W_ref))
    assert apart > 0.2 * lr, apart                                 # the two losses lead to clearly different weights ...
    assert err <= 0.02 * lr, (err, apart)                          # ... and the library follows the soft one


# ---- 8. input checks ---------------------------------------------------------------------------------------------------------------
def test_null_cotangent_is_rejected_before_any_launch():
    import scone_gcn_b200 as sg
    from scone_gcn_b200._lib import SconeError, check, lib
    ds, cx, net, W = scone_setup('scone', [16, 16, 16], 16, 0.1)
    ptr, fe, fv = sg.flows_to_csr(ds.flows)
    last = ds.last_nodes.astype(np.int32)
    assert net.plan(ptr, fe, fv, last)
    dev = [torch.as_tensor(a, device='cuda') for a in (ptr, fe, fv, last)]
    dptr = [C.c_void_p(t.data_ptr()) for t in dev]
    hptr = [a.ctypes.data_as(C.c_void_p) for a in (ptr, fe, fv, last)]
    p = dataset_problem('small')
    bunch = p.model([8, 8], micro_batch=16)
    bptr = [a.ctypes.data_as(C.c_void_p) for a in (*p.csr(), np.ascontiguousarray(p.last_nodes, np.int32))]
    L = lib()
    calls = {
        'scone_model_vjp_dev': lambda: L.scone_model_vjp_dev(net.handle, ds.n_traj, *dptr, None, 1.0, 1, None),
        'scone_model_vjp_host': lambda: L.scone_model_vjp_host(net.handle, ds.n_traj, *hptr, None, 1.0, 1, None),
        'scone_model_vjp_planned_dev': lambda: L.scone_model_vjp_planned_dev(net.handle, 4, None, None, 1.0, 1, None),
        'scone_model_vjp_planned_host': lambda: L.scone_model_vjp_planned_host(net.handle, 4, None, None, 1.0, 1, None),
        'scone_bunch_vjp_host': lambda: L.scone_bunch_vjp_host(bunch.handle, p.B, *bptr, None, 1.0, 1, None),
    }
    torch.cuda.synchronize()
    for name, call in calls.items():
        before = L.scone_launch_count()
        with pytest.raises(SconeError, match='code 2'):
            check(call(), name)
        assert L.scone_launch_count() == before, name

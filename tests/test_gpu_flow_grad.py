"""Gradient of the log-probs with respect to the flow values (scone_model_vjp_flows_*, SconeModel.vjp_flows, the flow_val input of
scone_gcn_b200.torch_ops.logprobs): dflow[p] = d(sum cot * logprob) / d flow_val[p] at every CSR entry of the batch.

  - against torch.autograd.grad of the float64 oracle with respect to its dense flows, gathered at the CSR entries, on every pipeline,
    the hash plan, the BIG launch and high-degree complexes;
  - zero-valued entries inside the readout cone whose neighbourhood carries no other flow (their gradient reads rows a non-zero value
    would make live), entries outside the cone (exactly 0), edge ids out of range (0) and empty trajectories;
  - the [grads | nll_sum | count] buffer is vjp()'s bit for bit; _host equals _dev; runs and micro-batch sizes give the same dflow;
  - the torch op under a nonlinear loss through a learnable scale of the flows; NULL dflow / cot rejected before any launch.
Tolerances: dflow within 1e-4 of the largest |dflow_ref| (the suite's style for gradients); the buffer meets check_buffer's."""
import ctypes as C

import numpy as np
import pytest
import torch

from golden_util import Dataset
from oracle import scone_oracle as so
from test_gpu_high_degree import fused_net, problem, scaled_weights
from test_gpu_vjp import CASES, check_buffer, random_cot, scone_setup

pytestmark = pytest.mark.gpu


def oracle_flow_vjp(model, B1, B2, last, flows, W, cot):
    """(logprobs, sum cot * lp, [d/dW], d/dflows [B, E]) of the float64 oracle with the dense flows as a differentiable input."""
    B = len(last)
    orc = so.DenseOracle(model, so.shift_matrices(B1, B2, model), B1, last, flows, np.zeros((B, 1)), dtype=torch.float64)
    F = orc.flows.clone().requires_grad_(True)
    orc.flows = F
    Wt = [torch.as_tensor(np.asarray(w, np.float64)).requires_grad_(True) for w in W]
    lp = orc.forward(Wt)[:, :, 0]
    ell = (lp * torch.as_tensor(np.asarray(cot, np.float64))).sum()
    g = torch.autograd.grad(ell, Wt + [F])
    return lp.detach().numpy(), float(ell.detach()), [x.numpy() for x in g[:-1]], g[-1].numpy()[:, :, 0]


def gather(dF, ptr, fe):
    """dF [B, E] at the CSR entries; an edge id out of range gets 0."""
    out = np.zeros(len(fe))
    E = dF.shape[1]
    for t in range(len(ptr) - 1):
        for p in range(ptr[t], ptr[t + 1]):
            if 0 <= fe[p] < E:
                out[p] = dF[t, fe[p]]
    return out


def check_dflow(got, ref, what):
    assert got.shape == ref.shape and np.isfinite(got).all(), what
    scale = float(np.abs(ref).max())
    assert scale > 0, what
    assert np.abs(got - ref).max() <= 1e-4 * scale, (what, np.abs(got - ref).max(), scale)


def make_net(model, hidden, mb, scale, variant, monkeypatch, seed=0):
    if variant == 'hash':
        monkeypatch.setenv('SCONE_FUSED_TABLE', '0')                  # read when a model is created
    ds, cx, net, W = scone_setup(model, hidden, mb, scale, seed)
    monkeypatch.delenv('SCONE_FUSED_TABLE', raising=False)
    if isinstance(variant, int) and variant != net.pipeline:
        net.set_pipeline(variant)
    assert net.pipeline == (variant if isinstance(variant, int) else 4)
    if variant == 'hash':
        assert net.fused_info()['table_plan_mb'] == 0
    return ds, cx, net, W


# ---- 1. against the float64 oracle -----------------------------------------------------------------------------------------------
FLOW_CASES = [c[:3] + (c[4], None) for c in CASES if not c[3]] + [('scone', [16, 16, 16], 1, 0.1, 1), ('scone', [32, 32, 32], 2, 0.1, 2),
                                                                  ('scone', [16, 16, 16], 4, 0.1, 'hash')]


@pytest.mark.parametrize('model,hidden,pipeline,scale,variant', FLOW_CASES,
                         ids=['%s-%s-p%d%s' % (c[0], 'x'.join(map(str, c[1])), c[2], '' if c[4] is None else '-%s' % c[4]) for c in FLOW_CASES])
def test_flow_gradient_matches_the_float64_oracle(model, hidden, pipeline, scale, variant, monkeypatch):
    import scone_gcn_b200 as sg
    ds, cx, net, W = make_net(model, hidden, 16, scale, pipeline if variant is None else variant, monkeypatch)
    assert net.pipeline == pipeline
    rs = np.random.RandomState(len(hidden) + hidden[0] + 1)
    B = ds.n_traj
    cot = random_cot(rs, B, cx.D)
    ptr, fe, fv = sg.flows_to_csr(ds.flows)
    lp_ref, ell, g_ref, dF = oracle_flow_vjp(model, ds.B1, ds.B2, ds.last_nodes, ds.flows, W, cot)
    buf, dflow = net.vjp_flows(ptr, fe, fv, ds.last_nodes, cot, 7.0)
    check_buffer(buf, net.n_params, net.unflatten, lp_ref, ell, g_ref, cot, 7.0, 'vjp_flows')
    check_dflow(dflow, gather(dF, ptr, fe), 'dflow')
    if model == 'ebli':                                            # the BIG launch (rows beyond the shared-memory store) took part
        whole = sg.SconeModel(cx, hidden, micro_batch=B)
        whole.set_weights(W)
        whole.forward(ptr, fe, fv, ds.last_nodes)
        assert max(int(whole.fused_header(t)[1:4].sum()) for t in range(B)) > net.fused_info()['cap_rows']


@pytest.mark.parametrize('name', ['wheel_72', 'hubs_8x120'])
def test_high_degree_flow_gradient_matches_the_oracle(name, monkeypatch):
    import scipy.sparse as sp
    hidden = [32, 32, 32]
    p = problem(name, 'scone', 3, seed=29)
    S = [sp.csr_matrix(m) for m in so.shift_matrices(p['B1'], p['B2'], 'scone')]
    W, _ = scaled_weights('scone', p['B1'], S, p['flows'][:, :, 0], p['last'], hidden, np.random.RandomState(11))
    B, D = len(p['last']), p['cx'].D
    cot = random_cot(np.random.RandomState(3), B, D)
    net = fused_net(monkeypatch, p, hidden, W, 'table', B)
    ptr, fe, fv = p['csr']
    lp_ref, ell, g_ref, dF = oracle_flow_vjp('scone', p['B1'], p['B2'], p['last'], p['flows'], W, cot)
    buf, dflow = net.vjp_flows(ptr, fe, fv, p['last'], cot, 5.0)
    check_buffer(buf, net.n_params, net.unflatten, lp_ref, ell, g_ref, cot, 5.0, name)
    check_dflow(dflow, gather(dF, ptr, fe), name)


# ---- 2. zero-valued, out-of-cone and out-of-range entries, empty trajectories ----------------------------------------------------
def augmented_batch(ds, model, W, rs):
    """The dataset plus two empty trajectories; every non-empty trajectory also gets, after its own entries: zero-valued entries
    inside the cone with no flow within two operator hops (the rows their gradient reads are live only if a zero value seeds
    liveness), zero-valued entries outside the readout cone T_0 (more than L operator hops from the edges the readout reads), and
    one edge id out of range.  Returns (ptr, fe, fv, last, dense flows, cot, dflow_ref, [(kind, p)])."""
    E = ds.flows.shape[1]
    flows = np.concatenate([ds.flows[:, :, 0], np.zeros((2, E))])
    last = np.concatenate([ds.last_nodes, ds.last_nodes[:2]]).astype(np.int32)
    B = len(last)
    cot = random_cot(rs, B, ds.D)
    _, _, _, dF = oracle_flow_vjp(model, ds.B1, ds.B2, last, flows, W, cot)
    S0, S1 = [np.abs(np.asarray(s)) for s in so.shift_matrices(ds.B1, ds.B2, model)]
    P = ((np.eye(E) + S0 + S1) > 0).astype(np.int32)
    P2 = (P @ P) > 0
    nb, _, _ = so.neighbourhood_tables(ds.B1, last)
    incident = np.abs(np.asarray(ds.B1)) > 0                       # [N, E]
    scale = np.abs(dF).max()
    ptr, fe, fv, kinds = [0], [], [], []
    for t in range(B):
        own = np.flatnonzero(flows[t])
        fe += list(own)
        fv += list(flows[t, own])
        if len(own):
            near = P2[:, own].any(axis=1)
            inside = np.flatnonzero(~near & (np.abs(dF[t]) > 0.02 * scale))
            cone = incident[nb[last[t]][nb[last[t]] >= 0]].any(axis=0)
            for _ in range(len(W) // 3):                           # one operator hop per layer: T_L -> T_0
                cone = (P @ cone.astype(np.int32)) > 0
            outside = np.flatnonzero(~cone & (flows[t] == 0))
            for kind, cand in (('zero-in-cone', inside[:2]), ('outside', outside[:2])):
                for e in cand:
                    kinds.append((kind, len(fe)))
                    fe.append(e)
                    fv.append(0.0)
            kinds.append(('out-of-range', len(fe)))
            fe.append(E + 3 if t % 2 else -2)
            fv.append(1.0)
        ptr.append(len(fe))
    ptr, fe, fv = np.asarray(ptr, np.int32), np.asarray(fe, np.int32), np.asarray(fv, np.float32)
    return ptr, fe, fv, last, flows, cot, gather(dF, ptr, fe), kinds


@pytest.mark.parametrize('variant', ['table', 'hash', 3, 0])
def test_zero_valued_and_out_of_cone_entries(variant, monkeypatch):
    ds, cx, net, W = make_net('scone', [16, 16, 16], 16, 0.1, variant, monkeypatch)
    ptr, fe, fv, last, flows, cot, ref, kinds = augmented_batch(ds, 'scone', W, np.random.RandomState(21))
    counts = {k: sum(1 for kk, _ in kinds if kk == k) for k in ('zero-in-cone', 'outside', 'out-of-range')}
    assert min(counts.values()) >= 3, counts
    _, dflow = net.vjp_flows(ptr, fe, fv, last, cot, 1.0)
    check_dflow(dflow, ref, 'augmented')
    for kind, p in kinds:
        if kind == 'zero-in-cone':
            assert abs(ref[p]) > 0.02 * np.abs(ref).max()          # a liveness seeded by value would leave these at 0
        else:
            assert dflow[p] == 0.0, (kind, p, dflow[p])
    # the weight buffer does not see the extra entries
    lp_ref, ell, g_ref, _ = oracle_flow_vjp('scone', ds.B1, ds.B2, last, flows, W, cot)
    buf = net.vjp(ptr, fe, fv, last, cot, 1.0)
    check_buffer(buf, net.n_params, net.unflatten, lp_ref, ell, g_ref, cot, 1.0, 'augmented buffer')


# ---- 3. the weight buffer, _host vs _dev, determinism, micro-batch independence -------------------------------------------------
@pytest.mark.parametrize('variant', ['table', 'hash', 3, 2, 1, 0])
def test_buffer_is_vjp_bit_for_bit_and_dflow_is_deterministic(variant, monkeypatch):
    import scone_gcn_b200 as sg
    from scone_gcn_b200._lib import check, lib
    ds, cx, net, W = make_net('scone', [16, 16, 16], 16, 0.2, variant, monkeypatch)
    ptr, fe, fv = sg.flows_to_csr(ds.flows)
    assert (fv != 0).all()
    cot = random_cot(np.random.RandomState(4), ds.n_traj, cx.D)
    ref = net.vjp(ptr, fe, fv, ds.last_nodes, cot, 3.0)
    runs = [net.vjp_flows(ptr, fe, fv, ds.last_nodes, cot, 3.0) for _ in range(2)]
    for buf, dflow in runs:
        assert np.array_equal(buf.view(np.uint32), ref.view(np.uint32))
        assert np.array_equal(dflow.view(np.uint32), runs[0][1].view(np.uint32))
    assert (runs[0][1] != 0).any()
    dev = [torch.as_tensor(a, device='cuda') for a in (ptr, fe, fv, ds.last_nodes.astype(np.int32), cot)]
    dflow = torch.full((len(fe),), 7.0, device='cuda')
    torch.cuda.synchronize()
    check(lib().scone_model_vjp_flows_dev(net.handle, ds.n_traj, *[C.c_void_p(t.data_ptr()) for t in dev], 3.0, 1,
                                          C.c_void_p(dflow.data_ptr()), None), 'scone_model_vjp_flows_dev')
    buf = net.read_grads()
    assert np.array_equal(buf.view(np.uint32), ref.view(np.uint32))
    assert np.array_equal(dflow.cpu().numpy().view(np.uint32), runs[0][1].view(np.uint32))
    # a sub-range of the batch overwrites its own entries only
    sub = np.full(len(fe), 5.0, np.float32)
    lo, hi = 7, 23
    a = [np.ascontiguousarray(x) for x in (ptr[lo:hi + 1], fe, fv, ds.last_nodes[lo:hi].astype(np.int32), cot[lo:hi])]
    check(lib().scone_model_vjp_flows_host(net.handle, hi - lo, *[x.ctypes.data_as(C.c_void_p) for x in a], 0.0, 1,
                                           sub.ctypes.data_as(C.c_void_p), None), 'scone_model_vjp_flows_host')
    inside = np.zeros(len(fe), bool)
    inside[ptr[lo]:ptr[hi]] = True
    assert (sub[~inside] == 5.0).all()
    check_dflow(sub[inside], runs[0][1][inside].astype(np.float64), 'sub-range')


def test_fused_dflow_does_not_depend_on_the_micro_batch():
    import scone_gcn_b200 as sg
    ds = Dataset('dataset_small.npz')
    cx = sg.SimplicialComplex.from_dense(ds.B1, ds.B2, 'scone')
    rs = np.random.RandomState(8)
    ptr, fe, fv = sg.flows_to_csr(ds.flows)
    cot = random_cot(rs, ds.n_traj, cx.D)
    out = []
    for mb in (7, 16, 64):
        net = sg.SconeModel(cx, [32, 32, 32], micro_batch=mb)
        assert net.pipeline == 4
        net.set_weights([(0.1 * np.random.RandomState(1).randn(*s)).astype(np.float32) for s in net.shapes])
        out.append(net.vjp_flows(ptr, fe, fv, ds.last_nodes, cot, 0.0)[1])
    for d in out[1:]:
        assert np.array_equal(d.view(np.uint32), out[0].view(np.uint32))


# ---- 4. the torch autograd op -----------------------------------------------------------------------------------------------------
def test_torch_op_flow_gradient_through_a_learnable_scale():
    import scone_gcn_b200 as sg
    from scone_gcn_b200 import torch_ops
    ds, cx, net, W = scone_setup('scone', [16, 16, 16], 32, 0.2)
    assert net.pipeline == 4
    dev = torch.device('cuda')
    ptr, fe, raw = sg.flows_to_csr(ds.flows)
    last = ds.last_nodes.astype(np.int32)
    ptr_t, fe_t, last_t = [torch.as_tensor(a, device=dev) for a in (ptr, fe, last)]
    raw_t = torch.as_tensor(raw, device=dev)
    q64 = np.random.RandomState(9).dirichlet(np.ones(cx.D), size=ds.n_traj)
    q = torch.as_tensor(q64, dtype=torch.float32, device=dev)

    def loss_of(lp, q):
        return (q * (torch.log(q) - lp)).sum() + 0.25 * (lp.exp() ** 2).sum()

    s = torch.tensor(1.3, device=dev, requires_grad=True)
    w = torch.as_tensor(net.flatten(W), device=dev).requires_grad_(True)
    flow_val = raw_t * s
    flow_val.retain_grad()
    loss = loss_of(torch_ops.logprobs(net, w, ptr_t, fe_t, flow_val, last_t), q)
    loss.backward()
    # float64 oracle with the same scale
    s64 = torch.tensor(1.3, dtype=torch.float64, requires_grad=True)
    orc = so.DenseOracle('scone', so.shift_matrices(ds.B1, ds.B2, 'scone'), ds.B1, ds.last_nodes, ds.flows, ds.targets, dtype=torch.float64)
    F = orc.flows.clone().requires_grad_(True)
    orc.flows = F * s64
    Wt = [torch.as_tensor(np.asarray(x, np.float64)).requires_grad_(True) for x in W]
    loss64 = loss_of(orc.forward(Wt)[:, :, 0], torch.as_tensor(q64))
    gs, gF, *gW = torch.autograd.grad(loss64, [s64, F] + Wt)
    ref = gather(gF.numpy()[:, :, 0] / 1.3, ptr, fe)              # d loss / d flow_val = (d loss / d F) / s
    assert abs(float(s.grad) - float(gs)) <= 1e-4 * float(np.abs(raw * ref).sum()), (float(s.grad), float(gs))
    check_dflow(flow_val.grad.cpu().numpy().astype(np.float64), ref, 'flow_val.grad')
    gmax = max(float(r.abs().max()) for r in gW)
    for i, (a, r) in enumerate(zip(net.unflatten(w.grad.cpu().numpy()), gW)):
        assert np.abs(a - r.numpy()).max() <= 1e-4 * max(float(r.abs().max()), 1e-3 * gmax), i
    # with flow_val not requiring grad the weight gradient is the one vjp_dev gives, bit for bit
    w2 = torch.as_tensor(net.flatten(W), device=dev).requires_grad_(True)
    g_plain, = torch.autograd.grad(loss_of(torch_ops.logprobs(net, w2, ptr_t, fe_t, (raw_t * 1.3).detach(), last_t), q), w2)
    assert torch.equal(g_plain, w.grad)


def test_torch_op_flow_gradient_on_an_empty_batch():
    from scone_gcn_b200 import torch_ops
    ds, cx, net, W = scone_setup('scone', [16, 16, 16], 32, 0.2)
    dev = torch.device('cuda')
    w = torch.as_tensor(net.flatten(W), device=dev).requires_grad_(True)
    i32 = lambda n: torch.zeros(n, dtype=torch.int32, device=dev)
    fv = torch.zeros(0, device=dev, requires_grad=True)
    lp = torch_ops.logprobs(net, w, i32(1), i32(0), fv, i32(0))
    gw, gf = torch.autograd.grad(lp.sum(), [w, fv])
    assert gf.shape == (0,) and not gw.any()


# ---- 5. input checks ---------------------------------------------------------------------------------------------------------------
def test_null_dflow_or_cotangent_is_rejected_before_any_launch():
    import scone_gcn_b200 as sg
    from scone_gcn_b200._lib import SconeError, check, lib
    ds, cx, net, W = scone_setup('scone', [16, 16, 16], 16, 0.1)
    ptr, fe, fv = sg.flows_to_csr(ds.flows)
    last = ds.last_nodes.astype(np.int32)
    cot = np.zeros((ds.n_traj, cx.D), np.float32)
    out = np.zeros(len(fe), np.float32)
    dev = [torch.as_tensor(a, device='cuda') for a in (ptr, fe, fv, last, cot, out)]
    d = [C.c_void_p(t.data_ptr()) for t in dev]
    h = [a.ctypes.data_as(C.c_void_p) for a in (ptr, fe, fv, last, cot, out)]
    L = lib()
    calls = {
        'dev, NULL dflow': lambda: L.scone_model_vjp_flows_dev(net.handle, ds.n_traj, *d[:5], 1.0, 1, None, None),
        'dev, NULL cot': lambda: L.scone_model_vjp_flows_dev(net.handle, ds.n_traj, *d[:4], None, 1.0, 1, d[5], None),
        'host, NULL dflow': lambda: L.scone_model_vjp_flows_host(net.handle, ds.n_traj, *h[:5], 1.0, 1, None, None),
        'host, NULL cot': lambda: L.scone_model_vjp_flows_host(net.handle, ds.n_traj, *h[:4], None, 1.0, 1, h[5], None),
    }
    torch.cuda.synchronize()
    for name, call in calls.items():
        before = L.scone_launch_count()
        with pytest.raises(SconeError, match='code 2'):
            check(call(), name)
        assert L.scone_launch_count() == before, name

"""Pipeline 4 (trajectory-fused kernels, csrc/scone_fused.cu) through the C ABI: its integer plan against a NumPy / SciPy
restatement of cone & support, its results against the row-list pipeline and the oracle, determinism, chunking, and the
big-trajectory variant (rows in global scratch)."""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

from golden_util import Dataset, load, weights_of
from oracle import scone_oracle as so

pytestmark = pytest.mark.gpu


def cpu_live_rows(cx, n_layers, flows_row, last):
    """Live rows per layer (sets of caller edge ids) for one trajectory: receptive cone of the readout intersected layer by layer
    with the structural support of the flows (DESIGN.md: cone & support)."""
    E = cx.E
    pats = []
    for k in range(2):
        rowptr, col, val = cx.shift_csr(k)
        pats.append(sp.csr_matrix((np.ones(len(col)), col, rowptr), shape=(E, E)))
    pat = ((pats[0] + pats[1] + sp.identity(E, format='csr')) > 0).astype(np.int32).tocsr()
    nb = cx.nbrhoods[last]
    nb = nb[nb >= 0]
    en = cx._edge_nodes
    top = np.zeros(E, bool)
    for v in nb:
        top |= (en[:, 0] == v) | (en[:, 1] == v)
    cones = [None] * (n_layers + 1)
    cones[n_layers] = top
    for l in range(n_layers - 1, 0, -1):
        cones[l] = (pat @ cones[l + 1].astype(np.int32)) > 0
    live = [None, cones[1] & ((pat @ (flows_row != 0).astype(np.int32)) > 0)]
    for l in range(2, n_layers + 1):
        live.append(cones[l] & ((pat @ live[l - 1].astype(np.int32)) > 0))
    return live


@pytest.fixture(params=['table', 'hash'])
def plan_kind(request, monkeypatch):
    """Both plan kernels: the table plan (csrc/scone_plan_table.cu, the default) and the hash plan (SCONE_FUSED_TABLE=0, its fallback)."""
    monkeypatch.setenv('SCONE_FUSED_TABLE', '1' if request.param == 'table' else '0')      # read when a model is created
    return request.param


def check_plan_kind(net, plan_kind):
    assert (net.fused_info()['table_plan_mb'] > 0) == (plan_kind == 'table')


@pytest.mark.parametrize('model,hidden', [('scone', [16, 16, 16]), ('scone', [32, 32]), ('ebli', [16, 16, 16]), ('scone', [32])])
def test_plan_live_rows_match_cpu_sets(model, hidden, plan_kind):
    import scone_gcn_b200 as sg
    ds = Dataset('dataset_small.npz')
    cx = sg.SimplicialComplex.from_dense(ds.B1, ds.B2, model)
    B = 24
    net = sg.SconeModel(cx, hidden, micro_batch=B)
    assert net.pipeline == 4 and net.fused_info() is not None
    check_plan_kind(net, plan_kind)
    rs = np.random.RandomState(0)
    net.set_weights([0.1 * rs.randn(*s) for s in net.shapes])
    ptr, fe, fv = sg.flows_to_csr(ds.flows[:B])
    net.forward(ptr, fe, fv, ds.last_nodes[:B])
    info = net.fused_info()
    for t in range(B):
        hdr = net.fused_header(t)
        live = cpu_live_rows(cx, len(hidden), ds.flows[t, :, 0], int(ds.last_nodes[t]))
        assert hdr[0] == 0
        for l in range(1, len(hidden) + 1):
            assert hdr[l] == int(live[l].sum()), (t, l, hdr[:4], [int(x.sum()) for x in live[1:]])
        assert max(hdr[1:4]) <= info['bound_list'] and hdr[11] <= info['bound_cone']


@pytest.mark.parametrize('model,hidden,mb,scale', [('scone', [16, 16, 16], 32, 0.1), ('scone', [32, 32, 32], 7, 0.1), ('ebli', [32, 32], 64, 0.02),
                                                   ('scone', [32], 16, 0.3), ('scone', [16, 16], 5, 0.3)])
def test_fused_matches_row_list_pipeline_and_is_deterministic(model, hidden, mb, scale, plan_kind):
    import scone_gcn_b200 as sg
    ds = Dataset('dataset_small.npz')
    cx = sg.SimplicialComplex.from_dense(ds.B1, ds.B2, model)
    ptr, fe, fv = sg.flows_to_csr(ds.flows)
    net = sg.SconeModel(cx, hidden, micro_batch=mb)
    assert net.pipeline == 4
    check_plan_kind(net, plan_kind)
    rs = np.random.RandomState(len(hidden) * 10 + mb)
    net.set_weights([scale * rs.randn(*s_) for s_ in net.shapes])
    mask = (rs.rand(ds.n_traj) < 0.7).astype(np.float32)
    out = {}
    for which in (4, 3, 4, 0):
        net.set_pipeline(which)
        lp = net.forward(ptr, fe, fv, ds.last_nodes)
        buf = net.loss_grad(ptr, fe, fv, ds.last_nodes, ds.raw['targets_argmax'], mask)
        if which in out:                                              # run-to-run: bit for bit
            assert np.array_equal(out[which][0], lp) and np.array_equal(out[which][1], buf)
        out[which] = (lp, buf)
    n = net.n_params
    for ref in (3, 0):
        assert np.abs(out[4][0] - out[ref][0]).max() <= 1e-5 * max(1.0, np.abs(out[ref][0]).max())
        assert out[4][1][n + 1] == out[ref][1][n + 1] == mask.sum()
        assert abs(out[4][1][n] - out[ref][1][n]) <= 1e-5 * max(1.0, abs(out[ref][1][n]))
        off = 0
        gmax = np.abs(out[ref][1][:n]).max()
        for shp in net.shapes:
            k = shp[0] * shp[1]
            a, r = out[4][1][off:off + k], out[ref][1][off:off + k]
            assert np.abs(a - r).max() <= 1e-4 * max(np.abs(r).max(), 1e-3 * gmax), (ref, shp)
            off += k


def test_fused_results_do_not_depend_on_chunking():
    import scone_gcn_b200 as sg
    ds = Dataset('dataset_small.npz')
    fx = load('model_small_scone_h16.npz')
    cx = sg.SimplicialComplex.from_dense(ds.B1, ds.B2, 'scone')
    ptr, fe, fv = sg.flows_to_csr(ds.flows)
    W = weights_of(fx, 'w_big')
    outs, grads = [], []
    for mb in (ds.n_traj, 5, 1):
        net = sg.SconeModel(cx, [16, 16, 16], micro_batch=mb)
        assert net.pipeline == 4
        net.set_weights(W)
        outs.append(net.forward(ptr, fe, fv, ds.last_nodes))
        grads.append(net.loss_grad(ptr, fe, fv, ds.last_nodes, ds.raw['targets_argmax'], np.ones(ds.n_traj, np.float32)))
    assert np.array_equal(outs[0], outs[1]) and np.array_equal(outs[0], outs[2])    # per-trajectory log-probs: bit for bit
    for g in grads[1:]:
        assert np.abs(g - grads[0]).max() <= 1e-5 * np.abs(grads[0]).max()
    assert np.abs(outs[0] - fx['big_logprobs'][:, :, 0]).max() < 1e-5                # and they are the reference's


def test_fused_big_trajectories_use_the_global_row_store(plan_kind):
    """ebli on the small complex: three L1^2 hops cover the whole complex, every layer has ~E live rows -> far more rows than the
    shared-memory store holds; the BIG variant must give the oracle's numbers."""
    import scone_gcn_b200 as sg
    ds = Dataset('dataset_small.npz')
    cx = sg.SimplicialComplex.from_dense(ds.B1, ds.B2, 'ebli')
    net = sg.SconeModel(cx, [32, 32, 32], micro_batch=16)
    assert net.pipeline == 4
    info = net.fused_info()
    rs = np.random.RandomState(2)
    W = [0.03 * rs.randn(*s) for s in net.shapes]
    net.set_weights(W)
    ptr, fe, fv = sg.flows_to_csr(ds.flows)
    lp = net.forward(ptr, fe, fv, ds.last_nodes)
    rows = [int(net.fused_header(t)[1:4].sum()) for t in range(min(16, ds.n_traj % 16 or 16))]
    assert max(rows) > info['cap_rows']                                              # the case this test is about
    orc = so.DenseOracle('ebli', so.shift_matrices(ds.B1, ds.B2, 'ebli'), ds.B1, ds.last_nodes, ds.flows, ds.targets, dtype=torch.float64)
    with torch.no_grad():
        ref = orc.forward(W).numpy()[:, :, 0]
    assert np.abs(lp - ref).max() <= 1e-5 * max(1.0, np.abs(ref).max())
    mask = ds.train_mask.astype(np.float32)
    buf = net.loss_grad(ptr, fe, fv, ds.last_nodes, ds.raw['targets_argmax'], mask)
    k = net.n_params
    _, g_ref = orc.loss_and_grads(W, ds.train_mask, 0.0)
    for a, r in zip(net.unflatten(buf[:k] / buf[k + 1]), g_ref):
        assert np.abs(a - r).max() <= 1e-4 * max(np.abs(r).max(), 1e-30)


def test_fused_mixed_trajectories_with_empty_flows_and_invalid_last_node(plan_kind):
    """Ragged inputs: a trajectory without flow entries (all logits 0 -> uniform log-probs over D slots) and one whose flows lie far
    from its last node, next to ordinary ones."""
    import scone_gcn_b200 as sg
    ds = Dataset('dataset_small.npz')
    cx = sg.SimplicialComplex.from_dense(ds.B1, ds.B2, 'scone')
    B = 12
    flows = ds.flows[:B].copy()
    flows[3] = 0.0
    last = ds.last_nodes[:B].copy()
    last[5] = ds.last_nodes[40]                                        # flows of trajectory 5, last node of trajectory 40
    net = sg.SconeModel(cx, [16, 16, 16], micro_batch=B)
    rs = np.random.RandomState(8)
    W = [0.3 * rs.randn(*s) for s in net.shapes]
    net.set_weights(W)
    ptr, fe, fv = sg.flows_to_csr(flows)
    lp = net.forward(ptr, fe, fv, last)
    assert np.allclose(lp[3], -np.log(cx.D), atol=1e-6)
    orc = so.DenseOracle('scone', so.shift_matrices(ds.B1, ds.B2, 'scone'), ds.B1, last, flows, ds.targets[:B], dtype=torch.float64)
    with torch.no_grad():
        ref = orc.forward(W).numpy()[:, :, 0]
    assert np.abs(lp - ref).max() <= 1e-5 * max(1.0, np.abs(ref).max())


def test_planned_set_gives_the_same_bits_as_planning_every_call(plan_kind):
    """scone_model_plan_* + *_planned_*: plan the dataset once, run batches by row index — bit-identical to the unplanned entry points
    (the same kernels on the same programs), for arbitrary row subsets in arbitrary order."""
    import scone_gcn_b200 as sg
    ds = Dataset('dataset_small.npz')
    fx = load('model_small_scone_h16.npz')
    cx = sg.SimplicialComplex.from_dense(ds.B1, ds.B2, 'scone')
    ptr, fe, fv = sg.flows_to_csr(ds.flows)
    net = sg.SconeModel(cx, [16, 16, 16], micro_batch=ds.n_traj)
    net.set_weights(weights_of(fx, 'w_big'))
    tgt = ds.raw['targets_argmax'].astype(np.int32)
    ref_lp = net.forward(ptr, fe, fv, ds.last_nodes)
    assert net.plan(ptr, fe, fv, ds.last_nodes)
    assert np.array_equal(net.forward_planned(), ref_lp)
    rs = np.random.RandomState(1)
    rows = rs.permutation(ds.n_traj)[:23]
    assert np.array_equal(net.forward_planned(rows), ref_lp[rows])
    mask = (rs.rand(len(rows)) < 0.8).astype(np.float32)
    got = net.loss_grad_planned(rows, tgt[rows], mask)
    from scone_gcn_b200.scone_trajectory_model import _Prepared
    sel = _Prepared([None, ds.last_nodes, (ptr, fe, fv)]).select(rows)
    ref = net.loss_grad(*sel, tgt[rows], mask)
    assert np.array_equal(got, ref)
    # an intervening unplanned call (its own chunk arena) does not disturb the set
    assert np.array_equal(net.forward_planned(rows), ref_lp[rows])


@pytest.mark.parametrize('model,hidden', [('scone', [32, 32, 32]), ('ebli', [16, 16]), ('scone', [16])])
def test_table_plan_and_hash_plan_write_the_same_plans(model, hidden, monkeypatch):
    """Headers (live rows per layer, pairs, cone entries, flow entries) equal, results bit-identical: same live sets, same row order,
    same entry order, same layer-1 scalars."""
    import scone_gcn_b200 as sg
    ds = Dataset('dataset_small.npz')
    cx = sg.SimplicialComplex.from_dense(ds.B1, ds.B2, model)
    ptr, fe, fv = sg.flows_to_csr(ds.flows)
    B = ds.n_traj
    rs = np.random.RandomState(5)
    out = {}
    W = None
    for kind in ('1', '0'):
        monkeypatch.setenv('SCONE_FUSED_TABLE', kind)
        net = sg.SconeModel(cx, hidden, micro_batch=B)
        assert net.pipeline == 4 and (net.fused_info()['table_plan_mb'] > 0) == (kind == '1')
        if W is None:
            W = [0.2 * rs.randn(*s_) for s_ in net.shapes]
        net.set_weights(W)
        lp = net.forward(ptr, fe, fv, ds.last_nodes)
        hdrs = np.stack([net.fused_header(t) for t in range(B)])
        buf = net.loss_grad(ptr, fe, fv, ds.last_nodes, ds.raw['targets_argmax'], np.ones(B, np.float32))
        out[kind] = (lp, hdrs, buf)
    assert np.array_equal(out['1'][1][:, [0, 1, 2, 3, 10, 11, 13]], out['0'][1][:, [0, 1, 2, 3, 10, 11, 13]])
    assert np.array_equal(out['1'][0], out['0'][0])
    assert np.array_equal(out['1'][2], out['0'][2])


@pytest.mark.parametrize('cuts,B', [(1, 1500), (6, 9000), (12, 17500)])
def test_host_entry_points_plan_in_parts_under_the_copy(cuts, B, plan_kind):
    """*_host entry points of a batch >= 512 trajectories: the flow arrays arrive on a copy stream in 1 / 2 / 4 parts (batches below
    8192 / below 16384 / larger); the first plan tier of a part runs when the part has landed, the later tiers once over all parts
    (table plan; the hash plan runs its tiers per part), one compute launch at the end — same bits as the device-pointer entry points."""
    import scone_gcn_b200 as sg
    from scone_gcn_b200 import _lib
    from scone_gcn_b200 import synthetic_data_gen as sdg
    sp = sdg.generate_sparse_dataset(4000, B, seed=3, n_waypoints=16, cuts_per_walk=cuts)
    assert sp.n_traj >= B
    cx = sg.SimplicialComplex.from_simplices(int(sp.n_nodes), sp.edges, sp.faces, 'scone')
    net = sg.SconeModel(cx, [16, 16, 16], micro_batch=B)
    assert net.pipeline == 4
    check_plan_kind(net, plan_kind)
    rs = np.random.RandomState(4)
    net.set_weights([0.3 * rs.randn(*s) for s in net.shapes])
    nnz = int(sp.traj_ptr[B])
    assert nnz >= 8192
    ptr, fe, fv = sp.traj_ptr[:B + 1].astype(np.int32), sp.flow_edge[:nnz].astype(np.int32), sp.flow_val[:nnz].astype(np.float32)
    last, tgt = sp.last_nodes[:B].astype(np.int32), sp.target_idx[:B].astype(np.int32)
    mask = (rs.rand(B) < 0.8).astype(np.float32)
    lp_host = net.forward(ptr, fe, fv, last)
    g_host = net.loss_grad(ptr, fe, fv, last, tgt, mask)
    d = {k: torch.from_numpy(v).cuda() for k, v in dict(ptr=ptr, fe=fe, fv=fv, last=last, tgt=tgt, mask=mask).items()}
    lp_dev = torch.empty(B, cx.D, device='cuda')
    L = _lib.lib()
    _lib.check(L.scone_model_forward_dev(net.handle, B, _lib.dptr(d['ptr']), _lib.dptr(d['fe']), _lib.dptr(d['fv']), _lib.dptr(d['last']),
                                         _lib.dptr(lp_dev), None), 'forward_dev')
    _lib.check(L.scone_model_loss_grad_dev(net.handle, B, _lib.dptr(d['ptr']), _lib.dptr(d['fe']), _lib.dptr(d['fv']), _lib.dptr(d['last']),
                                           _lib.dptr(d['tgt']), _lib.dptr(d['mask']), 1, None), 'loss_grad_dev')
    g_dev = net.read_grads()
    torch.cuda.synchronize()
    assert np.array_equal(lp_host, lp_dev.cpu().numpy())
    assert np.array_equal(g_host, g_dev)
    assert g_host[-1] == mask.sum()


def test_host_steps_enqueued_back_to_back_copy_under_the_previous_compute():
    """Three different batches through loss_grad_host + Adam + read_grads_async WITHOUT a host synchronisation in between (pinned host
    buffers): the flow arrays of step k + 1 are copied while step k computes (the staging buffers are free once step k's plan
    kernels are done).  Gradients of every step bit-identical to the same steps run one at a time with a synchronisation each."""
    import scone_gcn_b200 as sg
    from scone_gcn_b200 import synthetic_data_gen as sdg
    sp = sdg.generate_sparse_dataset(4000, 1500, seed=3, n_waypoints=16)
    cx = sg.SimplicialComplex.from_simplices(int(sp.n_nodes), sp.edges, sp.faces, 'scone')
    rs = np.random.RandomState(5)
    w0 = None
    batches = []
    for lo, hi in ((0, 700), (300, 1200), (700, 1500)):
        p0, p1 = int(sp.traj_ptr[lo]), int(sp.traj_ptr[hi])
        arrs = dict(ptr=(sp.traj_ptr[lo:hi + 1] - sp.traj_ptr[lo]).astype(np.int32), fe=sp.flow_edge[p0:p1].astype(np.int32),
                    fv=sp.flow_val[p0:p1].astype(np.float32), last=sp.last_nodes[lo:hi].astype(np.int32),
                    tgt=sp.target_idx[lo:hi].astype(np.int32), mask=(rs.rand(hi - lo) < 0.8).astype(np.float32))
        pins = {k: torch.from_numpy(v).pin_memory() for k, v in arrs.items()}
        batches.append({k: v.numpy() for k, v in pins.items()} | {'_keep': pins})

    def run(pipelined):
        nonlocal w0
        net = sg.SconeModel(cx, [16, 16, 16], micro_batch=2048)
        assert net.pipeline == 4
        if w0 is None:
            w0 = [0.3 * np.random.RandomState(6).randn(*s) for s in net.shapes]
        net.set_weights(w0)
        outs = []
        if pipelined:
            pinned = [torch.empty(net.n_params + 2, dtype=torch.float32).pin_memory() for _ in batches]
            for k, b in enumerate(batches):
                net.loss_grad(b['ptr'], b['fe'], b['fv'], b['last'], b['tgt'], b['mask'], zero_first=True, read=False)
                net.read_grads_async(pinned[k])
                net.adam_step(k, 1e-2, 5e-5)
            torch.cuda.synchronize()
            net.check_overflow()
            outs = [p.numpy().copy() for p in pinned]
        else:
            for k, b in enumerate(batches):
                outs.append(net.loss_grad(b['ptr'], b['fe'], b['fv'], b['last'], b['tgt'], b['mask'], zero_first=True))
                net.adam_step(k, 1e-2, 5e-5)
                torch.cuda.synchronize()
        return outs, net.get_weights()

    g_sync, w_sync = run(False)
    g_pipe, w_pipe = run(True)
    for a, b in zip(g_sync, g_pipe):
        assert np.array_equal(a, b)
    for a, b in zip(w_sync, w_pipe):
        assert np.array_equal(a, b)

"""High-degree complexes (D up to 128) through the C ABI against the float64 dense oracle.  Every complex elsewhere in the suite has
D <= 17; the code paths below exist only because of large degrees, and every test asserts that it reaches the one it is named for:
  - the fused compute kernel's shared-memory row store shrinks below 192 rows (hidden 32, D >= 72): trajectories split between the
    small and the BIG launch at cap_rows (scone_fused.cu, traj_smem_small / cap_rows);
  - readout pair lists longer than the 1024 entries the fused kernel stages (header word 10) and the row-list readout resolves from
    its table (kRoItems): hub endings of hubs_*;
  - softmax / dl / readout loops with more than one lane pass over the slots (D > 32), padded slots (logit 0, quirk Q1) dominating
    the normaliser: rim endings with 3 or 8 real slots out of up to 128;
  - unfused models of D > 32 start on the whole-support pipeline (2) instead of the cone pipeline (3);
  - the table plan at its degree limit and the hash plan next to it;
  - the degree limit itself: D = 129 is rejected when the model is created.
Tolerances are the suite's: log-probs 1e-5 * max(1, |ref|), mean NLL 1e-5 relative, weight gradients 1e-4 of their largest entry
(with the noise floor of test_gpu_tiny_complexes.py), masked counts exact."""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

from oracle import scone_oracle as so
from scone_gcn_b200._lib import SconeError
from test_index_tiny_complexes import CASES, HIGH_DEGREE, READOUT_PAIRS_STAGED, readout_pairs, wheel

pytestmark = pytest.mark.gpu

HIDDEN = [[16, 16, 16], [32, 32, 32], [32], [16]]
COMPLEXES = ['wheel_33', 'wheel_72', 'hubs_8x120', 'hubs_8x121']
FULL_ROW_STORE = 192                  # rows of the fused kernel's shared-memory store at hidden 32 when the degree leaves room for it
# Cases (complex, model, layers) at hidden 32 in which some trajectory has between cap_rows and 192 live rows.  In the others the totals
# jump over that band: one layer of wheel_72 has 144 rows in all; three layers of wheel_72 under scone, or of hubs_*, reach at least
# 226 / 2000 rows from a single flow edge; one ebli layer on hubs_8x121 goes from 121 rows straight past 192.
BAND_CASES = {('wheel_72', 'ebli', 3), ('hubs_8x120', 'scone', 1), ('hubs_8x121', 'scone', 1)}


def row_pattern(cx):
    """Pattern of I + S0 + S1 (caller's edge ids): the rows one layer reads."""
    pat = sp.identity(cx.E, format='csr')
    for k in range(2):
        rowptr, col, _ = cx.shift_csr(k)
        pat = pat + sp.csr_matrix((np.ones(len(col)), col, rowptr), shape=(cx.E, cx.E))
    return (pat > 0).astype(np.int32).tocsr()


def live_rows(cx, pat, n_layers, flows_row, last):
    """Live rows per layer of one trajectory (the restatement of cone & support of test_gpu_fused.cpu_live_rows): the receptive
    cone of the readout intersected layer by layer with the structural support of the flows."""
    nb = cx.nbrhoods[last]
    en = cx._edge_nodes
    top = np.isin(en[:, 0], nb[nb >= 0]) | np.isin(en[:, 1], nb[nb >= 0])
    cones = [None] * (n_layers + 1)
    cones[n_layers] = top
    for l in range(n_layers - 1, 0, -1):
        cones[l] = (pat @ cones[l + 1].astype(np.int32)) > 0
    live = [cones[1] & ((pat @ (flows_row != 0).astype(np.int32)) > 0)]
    for l in range(2, n_layers + 1):
        live.append(cones[l] & ((pat @ live[-1].astype(np.int32)) > 0))
    return [int(x.sum()) for x in live]


def find_band_flows(cx, n_layers, lo, hi, rs, tries=300):
    """Flows {-1, +1} and a last node whose live rows over all layers number in (lo, hi], or None: grows a connected edge set from a
    random seed edge in breadth-first order (the live sets only grow, by a few rows per edge near the seed) until the total passes lo."""
    pat = row_pattern(cx)
    nodes = np.unique(cx._edge_nodes)
    for _ in range(tries):
        last = int(rs.choice(nodes))
        seen = np.zeros(cx.E, bool)
        queue = [int(rs.randint(cx.E))]
        f = np.zeros(cx.E)
        while queue:
            e = queue.pop(0)
            if seen[e]:
                continue
            seen[e] = True
            f[e] = rs.choice([-1.0, 1.0])
            tot = sum(live_rows(cx, pat, n_layers, f, last))
            if tot > lo:
                if tot <= hi:
                    return f, last
                break
            queue += [int(x) for x in rs.permutation(pat.indices[pat.indptr[e]:pat.indptr[e + 1]]) if not seen[x]]
    return None


def act64(model, z):
    return np.tanh(z) if model == 'scone' else np.where(z >= 0, z, 0.01 * z)


def scaled_weights(model, B1, S, flows, last, hidden, rs, peak=2.0, logit_peak=3.0):
    """Random weights scaled layer by layer so that the float64 pre-activations of this batch peak at `peak` and its logits at
    `logit_peak`.  With S0 / S1 reaching entries of 126 (B2 B2^T of a hub edge) or 16641 (L1^2 under ebli) a fixed scale would either
    saturate every activation or leave it in the noise.  Returns the fp32 weights and the fp64 peaks they give."""
    Bt, E = flows.shape[:2]
    H = flows.reshape(Bt, E, 1).astype(np.float64)
    W, peaks = [], []

    def shift(Sk, H):                                                   # [E, E] @ [B, E, C] per trajectory
        c = H.shape[2]
        return (Sk @ H.transpose(1, 0, 2).reshape(E, -1)).reshape(E, Bt, c).transpose(1, 0, 2)
    cin = 1
    for c in hidden:
        w = [rs.randn(cin, c) for _ in range(3)]
        T = [H, shift(S[0], H), shift(S[1], H)]
        Z = sum(T[k] @ w[k] for k in range(3))
        s = peak / np.abs(Z).max()
        w = [(s * x).astype(np.float32) for x in w]
        Z = sum(T[k] @ w[k].astype(np.float64) for k in range(3))
        peaks.append(float(np.abs(Z).max()))
        H = act64(model, Z)
        W += w
        cin = c
    nb, _, B1_jax = so.neighbourhood_tables(B1, last)
    z = np.einsum('tde,tec->tdc', B1_jax[nb[last]], H)                # readout features of every slot
    wout = rs.randn(cin, 1)
    wout = (wout * logit_peak / np.abs(z @ wout).max()).astype(np.float32)
    W.append(wout)
    peaks.append(float(np.abs(z @ wout.astype(np.float64)).max()))
    return W, peaks


def problem(name, model, n_layers, seed, band=None, cx=None):
    """One batch on complex `name`, as the module docstring describes: dense {-1, 0, 1} flows ending at every hub (node of degree D)
    and at 8 rim nodes, flows on one or two edges only ending at the hubs, one trajectory without flows, and (band = (lo, hi)) one
    trajectory whose live rows over all layers number in (lo, hi].  Targets below n_nbrs, a mask with zeros."""
    import scone_gcn_b200 as sg
    n, edges, faces = CASES[name]
    edges, faces = np.asarray(edges, np.int64), np.asarray(faces, np.int64)
    B1, B2 = so.incidence_matrices(n, edges, faces)
    if cx is None:
        cx = sg.SimplicialComplex.from_simplices(n, edges, faces, model)
    deg = np.abs(B1).sum(axis=1).astype(int)
    hubs, rim = np.flatnonzero(deg == cx.D), np.flatnonzero(deg < cx.D)
    rs = np.random.RandomState(seed)
    E = cx.E
    hub_rounds = max(1, 4 // len(hubs))
    rows, last = [], []
    for h in np.tile(hubs, hub_rounds):                                                   # dense flows: BIG trajectories
        rows.append(rs.choice([-1.0, 0.0, 1.0], size=E, p=[0.15, 0.7, 0.15]))
        last.append(h)
    for v in rs.choice(rim, 8, replace=False):
        rows.append(rs.choice([-1.0, 0.0, 1.0], size=E, p=[0.15, 0.7, 0.15]))
        last.append(v)
    for i, h in enumerate(np.tile(hubs, hub_rounds)):                                     # one or two edges: small trajectories
        f = np.zeros(E)
        f[rs.choice(E, 1 + i % 2, replace=False)] = rs.choice([-1.0, 1.0], size=1 + i % 2)
        rows.append(f)
        last.append(h)
    rows.insert(3, np.zeros(E))                                                            # no flows at all: every logit 0
    last.insert(3, hubs[0])
    band_t = None
    if band is not None:
        found = find_band_flows(cx, n_layers, band[0], band[1], rs)
        assert found is not None, ('no flows land in the band', name, model, n_layers, band)
        band_t = len(rows)
        rows.append(found[0])
        last.append(found[1])
    flows = np.stack(rows)[:, :, None]
    last = np.asarray(last, np.int64)
    nb, n_nbrs, _ = so.neighbourhood_tables(B1, last)
    tgt = np.array([rs.randint(0, k) for k in n_nbrs])
    targets = np.zeros((len(last), cx.D, 1))
    targets[np.arange(len(last)), tgt, 0] = 1.0
    mask = (rs.rand(len(last)) < 0.75).astype(np.float32)
    mask[[1, 4]] = [0.0, 1.0]
    return dict(cx=cx, B1=B1, B2=B2, last=last, flows=flows, targets=targets, tgt=tgt, mask=mask, n_nbrs=n_nbrs, band_t=band_t,
                csr=sg.flows_to_csr(flows), hubs=hubs)


class Oracle:
    """fp64 DenseOracle of one problem and weights: log-probs, mean NLL over the mask, weight gradients."""

    def __init__(self, p, model, W, dtype=torch.float64):
        self.orc = so.DenseOracle(model, so.shift_matrices(p['B1'], p['B2'], model), p['B1'], p['last'], p['flows'], p['targets'],
                                  dtype=dtype)
        W = [np.asarray(w, np.float64) for w in W]
        with torch.no_grad():
            self.lp = self.orc.forward(W).numpy()[:, :, 0]
        self.nll, self.grads = self.orc.loss_and_grads(W, p['mask'], 0.0)
        self.nll = float(self.nll)


def check_vs_oracle(net, p, ref, what, lp_tol=1e-5):
    """log-probs, mean NLL, masked count and weight gradients of one model / pipeline against the oracle; returns (lp, buf)."""
    ptr, fe, fv = p['csr']
    lp = net.forward(ptr, fe, fv, p['last'])
    assert np.isfinite(lp).all(), what
    err = np.abs(lp - ref.lp) / np.maximum(1.0, np.abs(ref.lp))
    assert err.max() <= lp_tol, (what, 'log-probs', float(err.max()))
    buf = net.loss_grad(ptr, fe, fv, p['last'], p['tgt'], p['mask'])
    k = net.n_params
    assert buf[k + 1] == p['mask'].sum(), what
    nll = buf[k] / buf[k + 1]
    assert abs(nll - ref.nll) <= 1e-5 * abs(ref.nll), (what, 'nll', nll, ref.nll)
    grads = net.unflatten(buf[:k] / buf[k + 1])
    gmax = max(np.abs(r).max() for r in ref.grads)
    for i, (a, r) in enumerate(zip(grads, ref.grads)):
        # an array whose true gradient is zero up to cancellation noise is held to the noise floor (test_gpu_tiny_complexes.py)
        assert np.abs(a - r).max() <= 1e-4 * max(np.abs(r).max(), 1e-3 * gmax, 1e-2), (what, 'grad', i, np.abs(a - r).max(), np.abs(r).max())
    return lp, buf


def run_twice(net, p):
    """(log-probs, gradient buffer) of two identical calls, asserted bit-identical."""
    ptr, fe, fv = p['csr']
    out = []
    for _ in range(2):
        out.append((net.forward(ptr, fe, fv, p['last']), net.loss_grad(ptr, fe, fv, p['last'], p['tgt'], p['mask'])))
    assert np.array_equal(out[0][0], out[1][0]) and np.array_equal(out[0][1], out[1][1])
    return out[0]


def fused_net(monkeypatch, p, hidden, W, kind, mb):
    """A model on the fused pipeline (4) with the table plan (kind 'table', the default) or the hash plan ('hash', its fallback)."""
    import scone_gcn_b200 as sg
    monkeypatch.setenv('SCONE_FUSED_TABLE', '1' if kind == 'table' else '0')                # read when a model is created
    net = sg.SconeModel(p['cx'], hidden, micro_batch=mb)
    monkeypatch.delenv('SCONE_FUSED_TABLE')
    assert net.pipeline == 4, (kind, hidden)
    assert (net.fused_info()['table_plan_mb'] > 0) == (kind == 'table')
    net.set_weights(W)
    return net


# The hash plan (the fused pipeline's fallback when the table plan does not fit, SCONE_FUSED_TABLE=0) reports a capacity overflow
# (code 4) on these hubs_* batches: its per-layer slot buffer is sized from the shared memory left next to its tables, and a live layer
# of a whole-complex cone needs more.  Reported, not silently wrong; the marks are strict, so they go when the capacity is raised.
HASH_PLAN_OVERFLOWS = pytest.mark.xfail(raises=SconeError, strict=True, reason='hash plan slot buffer overflows (code 4) on hubs_*')


@pytest.mark.parametrize('kind', ['table', 'hash'])
@pytest.mark.parametrize('model', ['scone', 'ebli'])
@pytest.mark.parametrize('hidden', HIDDEN, ids=lambda h: 'h' + 'x'.join(map(str, h)))
@pytest.mark.parametrize('name', COMPLEXES)
def test_fused_pipeline_matches_the_oracle_at_high_degree(name, hidden, model, kind, monkeypatch, request):
    """Pipeline 4 with the table plan or the hash plan against the fp64 oracle; the fused plan's live rows against the CPU
    restatement; bit-repeatable, independent of chunking, forward_planned bit-equal to forward."""
    import scone_gcn_b200 as sg
    if kind == 'hash' and name.startswith('hubs'):
        request.applymarker(HASH_PLAN_OVERFLOWS)
    L, C = len(hidden), hidden[0]
    D = HIGH_DEGREE[name][3]
    cx = sg.SimplicialComplex.from_simplices(*CASES[name], model)
    probe = sg.SconeModel(cx, hidden, micro_batch=8)
    cap = probe.fused_info()['cap_rows']
    del probe
    # hidden 32 at D >= 72: the fused row store is smaller than 192 rows.  A trajectory whose live rows number in (cap_rows, 192]
    # belongs to the BIG launch; a row count of 192 assumed anywhere in the small launch would go wrong exactly there.
    band = None
    if C == 32 and D >= 72:
        assert cap < FULL_ROW_STORE, cap
        if (name, model, L) in BAND_CASES:
            band = (cap, FULL_ROW_STORE)
    p = problem(name, model, L, seed=L * 7 + C + (model == 'ebli'), band=band, cx=cx)
    rs = np.random.RandomState(11)
    S = [sp.csr_matrix(m) for m in so.shift_matrices(p['B1'], p['B2'], model)]
    W, peaks = scaled_weights(model, p['B1'], S, p['flows'][:, :, 0], p['last'], hidden, rs)
    assert all(1.0 <= q <= 4.0 for q in peaks), peaks
    ref = Oracle(p, model, W)
    B = len(p['last'])
    mb = 7
    assert B % mb != 0
    ptr, fe, fv = p['csr']
    pat = row_pattern(cx)
    cpu_rows = np.array([live_rows(cx, pat, L, p['flows'][t, :, 0], p['last'][t]) for t in range(B)])

    net = fused_net(monkeypatch, p, hidden, W, kind, mb)
    lp, _ = check_vs_oracle(net, p, ref, (kind, 4))
    assert np.array_equal(run_twice(net, p)[0], lp)
    # the same batch in one chunk: every plan header readable, and chunking changes no bit
    whole = fused_net(monkeypatch, p, hidden, W, kind, B)
    info = whole.fused_info()
    assert info['chunk'] == B and info['cap_rows'] == cap
    assert np.array_equal(whole.forward(ptr, fe, fv, p['last']), lp)
    hdr = np.stack([whole.fused_header(t) for t in range(B)])
    assert np.array_equal(hdr[:, 1:L + 1], cpu_rows)
    rows = cpu_rows.sum(axis=1)
    assert (rows <= cap).any()
    if name.startswith('hubs') or band is not None:                                          # small and BIG in one launch
        assert (rows > cap).any()
    if band is not None:
        assert cap < rows[p['band_t']] <= FULL_ROW_STORE, (rows[p['band_t']], cap)
    if name.startswith('hubs'):                                                               # pair lists beyond the staged 1024
        assert (hdr[:, 10] > READOUT_PAIRS_STAGED).any() and (hdr[:, 10] <= READOUT_PAIRS_STAGED).any()
    assert whole.plan(ptr, fe, fv, p['last']) and np.array_equal(whole.forward_planned(), lp)


def unfused_problem(name, hidden, model):
    p = problem(name, model, len(hidden), seed=len(hidden) * 7 + hidden[0] + (model == 'ebli'))
    S = [sp.csr_matrix(m) for m in so.shift_matrices(p['B1'], p['B2'], model)]
    W, peaks = scaled_weights(model, p['B1'], S, p['flows'][:, :, 0], p['last'], hidden, np.random.RandomState(11))
    assert all(1.0 <= q <= 4.0 for q in peaks), peaks
    return p, W


@pytest.mark.parametrize('model', ['scone', 'ebli'])
@pytest.mark.parametrize('hidden', HIDDEN, ids=lambda h: 'h' + 'x'.join(map(str, h)))
@pytest.mark.parametrize('name', COMPLEXES)
def test_row_list_and_unit_pipelines_match_the_oracle_at_high_degree(name, hidden, model):
    """Pipelines 2, 1 and 0 (the default model of these widths is fused) against the fp64 oracle; 2 and 1 run the same arithmetic
    per row (bit-equal), every pipeline bit-repeatable.  On hubs_* the readouts resolve pair lists longer than their staged 1024."""
    import scone_gcn_b200 as sg
    p, W = unfused_problem(name, hidden, model)
    ref = Oracle(p, model, W)
    assert p['cx'].D == HIGH_DEGREE[name][3]
    mb = 7
    assert len(p['last']) % mb != 0
    net = sg.SconeModel(p['cx'], hidden, micro_batch=mb)
    net.set_weights(W)
    out = {}
    for which in (2, 1, 0):
        net.set_pipeline(which)
        check_vs_oracle(net, p, ref, which)
        out[which] = run_twice(net, p)
    assert np.array_equal(out[2][0], out[1][0])
    if name.startswith('hubs'):                                 # the row-list readout resolves pairs beyond kRoItems on the fly
        assert readout_pairs(p['B1'])[p['last']].max() > READOUT_PAIRS_STAGED


@pytest.mark.parametrize('model', ['scone', 'ebli'])
@pytest.mark.parametrize('name', COMPLEXES)
def test_forced_cone_pipeline_is_right_or_reports_overflow(name, model):
    """Pipeline 3 at D > 32 (not its default there): its 2048-edge cone staging either holds every trajectory — then the results are
    the oracle's — or the call fails with the overflow code (4).  Never silently wrong; after an overflow the same model gives the
    oracle's numbers on pipeline 2."""
    import scone_gcn_b200 as sg
    hidden = [16, 16, 16]
    p = problem(name, model, 3, seed=5)
    rs = np.random.RandomState(3)
    S = [sp.csr_matrix(m) for m in so.shift_matrices(p['B1'], p['B2'], model)]
    W, _ = scaled_weights(model, p['B1'], S, p['flows'][:, :, 0], p['last'], hidden, rs)
    ref = Oracle(p, model, W)
    net = sg.SconeModel(p['cx'], hidden, micro_batch=9)
    net.set_weights(W)
    net.set_pipeline(3)
    try:
        check_vs_oracle(net, p, ref, 3)
    except SconeError as e:
        assert '(code 4)' in str(e), str(e)
        net.set_pipeline(2)
        check_vs_oracle(net, p, ref, 2)


@pytest.mark.parametrize('name,pipeline', [('wheel_32', 3), ('wheel_33', 2)])
def test_four_layer_model_routing_at_the_degree_boundary(name, pipeline):
    """Unfused models (4 layers) start on the cone pipeline up to D = 32 and on the whole-support pipeline above; both match the oracle."""
    import scone_gcn_b200 as sg
    hidden = [16, 16, 16, 16]
    p = problem(name, 'scone', 4, seed=13)
    rs = np.random.RandomState(2)
    S = [sp.csr_matrix(m) for m in so.shift_matrices(p['B1'], p['B2'], 'scone')]
    W, _ = scaled_weights('scone', p['B1'], S, p['flows'][:, :, 0], p['last'], hidden, rs)
    net = sg.SconeModel(p['cx'], hidden, micro_batch=5)
    assert net.pipeline == pipeline and net.fused_info() is None
    net.set_weights(W)
    check_vs_oracle(net, p, Oracle(p, 'scone', W), pipeline)


@pytest.mark.parametrize('pipeline', [4, 2, 0])
def test_device_evaluation_at_high_degree(pipeline):
    """evaluate() (argmax choice, accuracy, NLL) and two_target_counts at D = 128 against NumPy on the returned log-probs: the
    argmax runs over 128 slots with the -100 masking beyond n_nbrs; counts exact."""
    import scone_gcn_b200 as sg
    hidden = [16, 16, 16]
    p = problem('hubs_8x121', 'scone', 3, seed=17)
    rs = np.random.RandomState(4)
    S = [sp.csr_matrix(m) for m in so.shift_matrices(p['B1'], p['B2'], 'scone')]
    W, _ = scaled_weights('scone', p['B1'], S, p['flows'][:, :, 0], p['last'], hidden, rs)
    net = sg.SconeModel(p['cx'], hidden, micro_batch=6)
    net.set_weights(W)
    net.set_pipeline(pipeline)
    ptr, fe, fv = p['csr']
    last, n_nbrs, tgt, mask = p['last'], p['n_nbrs'], p['tgt'], p['mask']
    lp = net.forward(ptr, fe, fv, last)
    masked = lp.copy()
    for i in range(len(masked)):
        masked[i, n_nbrs[i]:] = -100
    choice_ref = np.argmax(masked, axis=1)
    assert (choice_ref >= 32).any()                                                           # beyond the first lane pass
    got = net.evaluate(ptr, fe, fv, last, n_nbrs=n_nbrs, target_idx=tgt, mask=mask, want_choice=True, want_accuracy=True, want_nll=True)
    assert np.array_equal(got['choice'], choice_ref)
    assert got['accuracy'] == (int(((choice_ref == tgt) & (mask == 1)).sum()), int(mask.sum()))
    nll_ref = -(mask.astype(np.float64) * lp[np.arange(len(lp)), tgt]).sum()
    assert abs(got['nll'][0] - nll_ref) <= 1e-5 * abs(nll_ref) and got['nll'][1] == mask.sum()
    # the random other target: a different valid slot, and for two rows one beyond n_nbrs (counts as -100)
    rnd = np.array([(t + 1 + rs.randint(0, max(1, k - 1))) % max(k, 1) for t, k in zip(tgt, n_nbrs)])
    rnd[:2] = n_nbrs[:2]
    tv, rv = masked[np.arange(len(lp)), tgt], masked[np.arange(len(lp)), np.minimum(rnd, p['cx'].D - 1)]
    rv[:2] = -100.0
    m = mask == 1
    assert net.two_target_counts(tgt, rnd) == (int((tv > rv)[m].sum()), int((tv == rv)[m].sum()))


def test_saturated_logits_on_every_pipeline(monkeypatch):
    """scone, hubs_8x120, hidden 32 with saturated activations and logits beyond +-30: finite log-probs within tolerance of the fp64
    log-softmax on every pipeline (the normaliser's maximum subtraction carries the case)."""
    import scone_gcn_b200 as sg
    hidden = [32, 32, 32]
    p = problem('hubs_8x120', 'scone', 3, seed=23)
    rs = np.random.RandomState(6)
    S = [sp.csr_matrix(m) for m in so.shift_matrices(p['B1'], p['B2'], 'scone')]
    W, peaks = scaled_weights('scone', p['B1'], S, p['flows'][:, :, 0], p['last'], hidden, rs, peak=8.0, logit_peak=60.0)
    ref = Oracle(p, 'scone', W)
    # logits of the rows with padded slots (logit exactly 0): logit_j = lp_j - lp_pad
    pad = p['n_nbrs'] < p['cx'].D
    logits = ref.lp[pad] - ref.lp[pad, -1:]
    assert np.abs(logits).max() >= 30 and peaks[-1] >= 30
    # log-probs of -60 carry the fp32 rounding of logits of +-60: the same formulation in fp32 (DenseOracle) is measured here, and the
    # kernels may be at most twice as far from fp64 as it is
    lp32 = Oracle(p, 'scone', W, dtype=torch.float32).lp
    lp_tol = max(1e-5, 2 * float((np.abs(lp32 - ref.lp) / np.maximum(1.0, np.abs(ref.lp))).max()))
    assert lp_tol < 1e-4
    check_vs_oracle(fused_net(monkeypatch, p, hidden, W, 'table', 7), p, ref, ('table', 4), lp_tol)
    with pytest.raises(SconeError, match=r'\(code 4\)'):                                   # see HASH_PLAN_OVERFLOWS
        check_vs_oracle(fused_net(monkeypatch, p, hidden, W, 'hash', 7), p, ref, ('hash', 4), lp_tol)
    net = sg.SconeModel(p['cx'], hidden, micro_batch=7)
    net.set_weights(W)
    for which in (3, 2, 1, 0):
        net.set_pipeline(which)
        check_vs_oracle(net, p, ref, which, lp_tol)


def test_degree_above_the_limit_is_rejected_at_model_creation():
    """A wheel with 129 rim nodes (D = 129): the complex is accepted, a model on it is not, and the message names the limit."""
    import scone_gcn_b200 as sg
    n, edges, faces = wheel(129)
    cx = sg.SimplicialComplex.from_simplices(n, edges, faces, 'scone')
    assert cx.D == 129
    for hidden in ([16, 16, 16], [16, 16, 16, 16], [8]):
        with pytest.raises(SconeError, match='128'):
            sg.SconeModel(cx, hidden, micro_batch=4)
    # a valid model created right after it works
    p = problem('wheel_33', 'scone', 3, seed=29)
    rs = np.random.RandomState(8)
    S = [sp.csr_matrix(m) for m in so.shift_matrices(p['B1'], p['B2'], 'scone')]
    W, _ = scaled_weights('scone', p['B1'], S, p['flows'][:, :, 0], p['last'], [16, 16, 16], rs)
    net = sg.SconeModel(p['cx'], [16, 16, 16], micro_batch=7)
    net.set_weights(W)
    check_vs_oracle(net, p, Oracle(p, 'scone', W), 'after rejection')

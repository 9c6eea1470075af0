"""What happens after the gradient on the scone / ebli model: the Adam step (adam_kernel, csrc/scone_kernels.cu), the fused exchange + Adam
kernel of the data-parallel step run at one rank (dp_allreduce_adam_kernel, csrc/scone_dp.cu), and the capacity-overflow contract of
include/scone_b200.h (scone_model_check_overflow and the pipeline 2 / 3 notes):
  - while the device flag is set every Adam step leaves W, m and v untouched (the exchange kernel still writes the summed buffer back);
  - check_overflow, read_grads, forward_host, accuracy_host and eval_host report error code 4 once and clear the flag; the *_dev entry
    points, read_grads_async and adam_step never report it; eval_host leaves no log-probs for two_target_host after a report;
  - after a reported overflow the cone pipeline (3) gives the next batch bit for bit what a fresh model gives.

The Adam reference is oracle.adam_update (jax.experimental.optimizers.adam) in float64 on the buffer the kernel consumed:
g = grads / count + 2 wd W, b1 = 0.9, b2 = 0.999, eps = 1e-8, bias correction with i + 1.  The constants are the fp32 values the kernel
(and JAX on fp32 weights) uses.  m and v have no getter: they are observed through W over consecutive steps with different gradients,
the reference carrying its own float64 moments.

Two deterministic overflow triggers, each established on the CPU first; code 4 is a reported capacity condition, not a device fault:
  - the cone pipeline on fan_hub(128, 16): the readout cone of a trajectory ending at the hub has 2176 edges at its top level, beyond
    the 2048 cone edges per trajectory and level the cone kernel stages (kConeCap, csrc/scone_rows.cu);
  - the fused pipeline's hash plan (SCONE_FUSED_TABLE=0) on hubs_8x120: a live layer of a dense trajectory has more merged-row entries
    than its slot buffer can ever hold (the strict xfails of test_gpu_high_degree.py)."""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp
import torch

from golden_util import Dataset
from oracle import scone_oracle as so
from scone_gcn_b200._lib import SconeError
from test_gpu_high_degree import Oracle, check_vs_oracle, fused_net, problem, row_pattern, scaled_weights
from test_index_tiny_complexes import CASES

pytestmark = pytest.mark.gpu

U = 2.0 ** -24                                   # unit roundoff of fp32
B1F, B2F, EPSF = (float(np.float32(x)) for x in (0.9, 0.999, 1e-8))
LR = 1e-2
STEPS = (0, 1, 2, 100000)                        # 10^5: powf(b2, i + 1) underflows, both bias corrections are 1 in fp32
CONE_CAP = 2048                                  # cone edges per trajectory and level staged by the cone kernel (kConeCap)
CONE_HASH = 4096                                 # edges the cone kernel's per-level hash set holds (kConeHash)
HASH_SLOTS_MAX = 225 * 1024 // 2                 # the hash plan's slot buffer: at most half of its 225 KB of shared memory, 2 bytes a slot


# ---- Adam reference and tolerance -----------------------------------------------------------------------------------------------
def adam64(i, buf, W, m, v, lr, wd):
    """One step of oracle.adam_update in float64 from the fp32 weights W on the buffer [grads | nll_sum | count] the kernel consumed."""
    n = len(W)
    W = np.asarray(W, np.float64)
    g = buf[:n].astype(np.float64) / np.float64(buf[n + 1]) + 2.0 * float(np.float32(wd)) * W
    (x, m, v), = so.adam_update(i, [g], [(W, m, v)], float(np.float32(lr)), b1=B1F, b2=B2F, eps=EPSF, dtype=np.float64)
    return x, m, v


def adam_tol(i, W_prev, W_ref, lr):
    """Bound on |W_gpu - W_ref| for one step taken by both from the same fp32 W_prev, from fp32 rounding:
      - W - dW is rounded once (1/2 ulp) and dW is off by its own last rounding (1/2 ulp of W at most): 1 ulp(W_ref), doubled for an
        FMA the compiler may contract: 2 ulp(W_ref);
      - dW = lr * mhat / (sqrt(vhat) + eps) comes from g, m and v through about 12 rounded operations per step, each off by at most u
        relative to its larger operand; |mhat| / sqrt(vhat) is at most ~7 (Cauchy-Schwarz over the moment sums), so over the <= 4 steps
        of a sequence the moments carry at most 4 * 12 * 7 u lr ~ 2e-5 lr;  the measured errors sit far below (printed as err/tol);
      - c = 1 - powf(b, i + 1) is rounded in fp32: powf is within 4 ulp, and the subtraction cancels, so c1 and c2 are off by
        4 u b^(i+1) / c relative (c2 under a square root: half of that) - |dW| (4 u b1^(i+1) / c1 + 2 u b2^(i+1) / c2).
    A wrong weight-decay factor, a bias correction with i instead of i + 1 or a skipped / repeated moment update moves W by a sizeable
    fraction of lr: far outside."""
    dW = np.abs(np.asarray(W_prev, np.float64) - W_ref)
    ulp = np.spacing(np.abs(W_ref).astype(np.float32)).astype(np.float64)
    c1, c2 = 1.0 - B1F ** (i + 1), 1.0 - B2F ** (i + 1)
    bias = 4 * U * B1F ** (i + 1) / c1 + 2 * U * B2F ** (i + 1) / c2
    return 2 * ulp + 2e-5 * lr + dW * bias


def check_step(got, W_prev, W_ref, i, lr, what):
    """Asserts one step against the reference and returns the worst err / tol."""
    err = np.abs(got.astype(np.float64) - W_ref)
    tol = adam_tol(i, W_prev, W_ref, lr)
    assert np.isfinite(got).all(), what
    worst = int(np.argmax(err / tol))
    assert (err <= tol).all(), (what, 'step', i, 'entry', worst, float(err[worst]), float(tol[worst]), float(got[worst]), W_ref[worst])
    return float((err / tol).max())


def weights(net):
    """Flat fp32 weights (synchronous copy)."""
    return net.flatten(net.get_weights())


def device_buffer(net):
    torch.cuda.synchronize()
    return net.grads_tensor().cpu().numpy().copy()


def write_buffer(net, buf):
    """Writes a chosen [grads | nll_sum | count] into the model's device buffer (exact inputs for the step)."""
    assert buf.dtype == np.float32 and buf.shape == (net.n_params + 2,)
    net.grads_tensor().copy_(torch.from_numpy(buf).cuda())
    torch.cuda.synchronize()


def chosen_buffer(n, count, rs, zeros=(), neg_zeros=()):
    """grads / count spread over two decades with random signs; entries `zeros` exactly 0, `neg_zeros` exactly -0.0."""
    t = rs.choice([-1.0, 1.0], n) * 10.0 ** rs.uniform(-2, 0, n)
    buf = np.zeros(n + 2, np.float32)
    buf[:n] = (t * count).astype(np.float32)
    buf[list(zeros)] = 0.0
    buf[list(neg_zeros)] = -0.0
    buf[n] = np.float32(rs.uniform(10, 100))
    buf[n + 1] = np.float32(count)
    return buf


def unit_model(hidden):
    """A model of any widths (pipeline 0 accepts them all) on a one-triangle complex: only its weights and buffers are used."""
    import scone_gcn_b200 as sg
    cx = sg.SimplicialComplex.from_simplices(*CASES['single_triangle'], 'scone')
    return sg.SconeModel(cx, list(hidden), micro_batch=4)


def initial_weights(net, rs):
    return (rs.choice([-1.0, 1.0], net.n_params) * rs.uniform(0.05, 1.0, net.n_params)).astype(np.float32)


# model sizes: n_params = 32 (one 256-thread block), 224 (one block, nearly full), 6304 (25 blocks, ragged tail of 160), 18656 (73 blocks,
# ragged tail of 224)
ADAM_SIZES = [(8,), (8, 8), (32, 64), (64, 64, 32)]
COUNTS = (37.0, 12.0, 5.0, 37.0)                 # masked-row counts of the four steps: none a power of two


@pytest.mark.parametrize('wd', [0.0, 5e-5, 0.1])
@pytest.mark.parametrize('hidden', ADAM_SIZES, ids=lambda h: 'h' + 'x'.join(map(str, h)))
def test_adam_steps_match_float64_adam(hidden, wd):
    """Steps 0, 1, 2 and 10^5 with different chosen gradients (exact zeros among them) against the float64 restatement.  With wd = 0.1 the
    ridge term is as large as the data term; with wd = 0 an entry whose gradient is exactly 0 at every step keeps its weight bit for bit."""
    net = unit_model(hidden)
    n = net.n_params
    assert (n <= 256) == (hidden in [(8,), (8, 8)]) and (n <= 256 or n % 256 != 0)
    rs = np.random.RandomState(n + int(wd * 1e6))
    W = initial_weights(net, rs)
    net.set_weights(net.unflatten(W))
    zeros = np.arange(3, n, 7)
    m = v = np.zeros(n)
    worst = 0.0
    for i, count in zip(STEPS, COUNTS):
        buf = chosen_buffer(n, count, rs, zeros=zeros)
        write_buffer(net, buf)
        net.adam_step(i, LR, wd)
        got = weights(net)
        W_ref, m, v = adam64(i, buf, W, m, v, LR, wd)
        worst = max(worst, check_step(got, W, W_ref, i, LR, (hidden, wd)))
        if wd == 0.0:
            assert np.array_equal(got[zeros].view(np.uint32), W[zeros].view(np.uint32))      # update exactly 0.0
        assert np.array_equal(device_buffer(net), buf)                                            # the step reads the buffer only
        W = got
    print('adam %s wd=%g: worst err/tol %.3g' % (hidden, wd, worst))


def test_adam_steps_from_a_real_gradient():
    """End to end on dataset_small: loss_grad, then Adam on the buffer it left, three steps, against the float64 restatement."""
    import scone_gcn_b200 as sg
    ds = Dataset('dataset_small.npz')
    cx = sg.SimplicialComplex.from_dense(ds.B1, ds.B2, 'scone')
    net = sg.SconeModel(cx, [16, 16], micro_batch=32)
    rs = np.random.RandomState(5)
    net.set_weights([0.3 * rs.randn(*s) for s in net.shapes])
    W = weights(net)
    ptr, fe, fv = sg.flows_to_csr(ds.flows)
    tgt = ds.raw['targets_argmax'].astype(np.int32)
    m = v = np.zeros(net.n_params)
    worst = 0.0
    for i in range(3):
        mask = (rs.rand(ds.n_traj) < 0.6).astype(np.float32)
        buf = net.loss_grad(ptr, fe, fv, ds.last_nodes, tgt, mask)
        assert buf[-1] == mask.sum() and np.abs(buf[:-2]).max() > 0
        net.adam_step(i, LR, 5e-5)
        got = weights(net)
        W_ref, m, v = adam64(i, buf, W, m, v, LR, 5e-5)
        worst = max(worst, check_step(got, W, W_ref, i, LR, 'dataset_small'))
        W = got
    print('adam dataset_small: worst err/tol %.3g' % worst)


def test_set_weights_resets_and_keep_state_keeps_the_moments():
    """After two steps: set_weights_keep_state continues from the moments, set_weights starts again from zero moments."""
    n_steps = 2
    wd = 0.1
    out = {}
    for keep in (True, False):
        net = unit_model((32, 64))
        n = net.n_params
        rs = np.random.RandomState(9)
        W = initial_weights(net, rs)
        net.set_weights(net.unflatten(W))
        m = v = np.zeros(n)
        for i in range(n_steps):
            buf = chosen_buffer(n, COUNTS[i], rs)
            write_buffer(net, buf)
            net.adam_step(i, LR, wd)
            W_ref, m, v = adam64(i, buf, W, m, v, LR, wd)
            got = weights(net)
            check_step(got, W, W_ref, i, LR, 'before set_weights')
            W = got
        W2 = np.float32(0.5) * W
        net.set_weights(net.unflatten(W2), reset_adam=not keep)
        torch.cuda.synchronize()
        if not keep:
            m = v = np.zeros(n)
        buf = chosen_buffer(n, COUNTS[n_steps], rs)
        write_buffer(net, buf)
        net.adam_step(n_steps, LR, wd)
        got = weights(net)
        W_ref, _, _ = adam64(n_steps, buf, W2, m, v, LR, wd)
        check_step(got, W2, W_ref, n_steps, LR, ('keep' if keep else 'reset'))
        out[keep] = got
    assert np.abs(out[True] - out[False]).max() > 0.1 * LR                      # the two states give visibly different steps


# ---- the fused exchange + Adam kernel at one rank -----------------------------------------------------------------------------------
def dp_create(n_floats):
    import scone_gcn_b200 as sg
    h = C.c_void_p()
    rc = sg.lib().scone_dp_create(0, 1, int(n_floats), C.byref(h))
    return rc, h


def dp_step(net, dp, i, lr, wd):
    import scone_gcn_b200 as sg
    return sg.lib().scone_model_dp_adam_step(net.handle, dp, int(i), float(lr), float(wd), None)


def dp_slices(n):
    """(blocks, floats per block) of dp_allreduce_adam_kernel over n = n_params + 2 floats (scone_dp_create)."""
    nb = min(-(-n // 256), 64)
    return nb, -(-n // nb)


# (hidden, the slicing case it reaches).  nll_sum and count always share the last block: per = ceil(n / nb) leaves that block at least
# per - nb + 1 >= 2 floats for every n (nb = 1: n >= 3; nb < 64: per > 128 > nb; nb = 64: per > 256), so no model size separates them.
DP_SIZES = [((8,), 'one block'), ((64,), 'two blocks, the scalars after 127 gradients'), ((64, 64, 32), '64-block cap, per > 256')]


@pytest.mark.parametrize('hidden,case', DP_SIZES, ids=[c.split(',')[0] for _, c in DP_SIZES])
def test_exchange_kernel_at_one_rank_matches_the_adam_step(hidden, case):
    """scone_model_dp_adam_step at world 1 against scone_model_adam_step on a twin model: bit-identical weights over five steps (both
    parities of the sequence number), the buffer written back as the one-rank sum 0 + x (-0.0 reads back as +0.0), status 0; a handle
    created for another size is refused with code 2 and changes nothing."""
    import scone_gcn_b200 as sg
    a, b = unit_model(hidden), unit_model(hidden)
    n = a.n_params
    nb, per = dp_slices(n + 2)
    last = n + 2 - (nb - 1) * per
    if case == 'one block':
        assert nb == 1
    elif case.startswith('two blocks'):
        assert nb == 2 and per < 256 and n // per == 1 and last == 129 and last - 2 == 127
    else:
        assert nb == 64 and per > 256 and last < per
    assert n // per == (n + 1) // per == nb - 1
    rs = np.random.RandomState(n)
    W = initial_weights(a, rs)
    a.set_weights(a.unflatten(W))
    b.set_weights(b.unflatten(W))
    rc, dp = dp_create(n + 2)
    assert rc == 0, sg.lib().scone_last_error()
    try:
        wd = 0.1
        m = v = np.zeros(n)
        for k, i in enumerate(STEPS + (100001,)):
            negz = np.arange(5, n, 11)
            buf = chosen_buffer(n, COUNTS[k % 4], rs, zeros=np.arange(2, n, 13), neg_zeros=negz)
            write_buffer(a, buf)
            write_buffer(b, buf)
            a.adam_step(i, LR, wd)
            assert dp_step(b, dp, i, LR, wd) == 0
            wa, wb = weights(a), weights(b)
            assert np.array_equal(wa.view(np.uint32), wb.view(np.uint32)), (case, 'step', i, np.flatnonzero(wa != wb)[:8])
            W_ref, m, v = adam64(i, buf, W, m, v, LR, wd)
            check_step(wb, W, W_ref, i, LR, (case, 'dp'))
            W = wb
            back = device_buffer(b)
            assert np.array_equal(back, buf) and not np.signbit(back[negz]).any()          # written back, as the sum 0 + x
            assert np.array_equal(device_buffer(a).view(np.uint32), buf.view(np.uint32))   # the plain step only reads it
        assert sg.lib().scone_dp_status(dp, None) == 0
        for wrong in (n + 1, n + 3):
            rc, bad = dp_create(wrong)
            assert rc == 0
            try:
                assert dp_step(b, bad, 0, LR, wd) == 2
                assert b'created for %d floats' % wrong in sg.lib().scone_last_error()
                assert np.array_equal(weights(b).view(np.uint32), W.view(np.uint32))
            finally:
                sg.lib().scone_dp_destroy(bad)
    finally:
        sg.lib().scone_dp_destroy(dp)


# ---- overflow triggers ------------------------------------------------------------------------------------------------------------
def fan_hub(n_rim, n_fan):
    """Hub 0 joined to rim nodes 1..n_rim; every rim node r carries its own fan: n_fan leaves joined to r, consecutive leaves joined,
    triangles (r, a, a + 1).  The hub has degree n_rim, a rim node 1 + n_fan, a leaf at most 3."""
    edges, faces, nxt = [], [], n_rim + 1
    for r in range(1, n_rim + 1):
        leaves = list(range(nxt, nxt + n_fan))
        nxt += n_fan
        edges += [(0, r)] + [(r, a) for a in leaves] + list(zip(leaves, leaves[1:]))
        faces += [(r, a, b) for a, b in zip(leaves, leaves[1:])]
    return nxt, sorted(edges), sorted(faces)


FAN_HIDDEN = [16, 16]


def cone_levels(cx, n_layers, last):
    """Edges of the readout cone of a trajectory ending at `last`, per cone-kernel level from the top (L - 1, listed) down to 0 (not
    listed): the edges incident to the neighbours of `last`, then one hop of I + S0 + S1 per level (the cone sets of test_gpu_fused)."""
    pat = row_pattern(cx)
    nb = cx.nbrhoods[last]
    en = cx._edge_nodes
    cur = np.isin(en[:, 0], nb[nb >= 0]) | np.isin(en[:, 1], nb[nb >= 0])
    out = [int(cur.sum())]
    for _ in range(n_layers - 1):
        cur = (pat @ cur.astype(np.int32)) > 0
        out.append(int(cur.sum()))
    return out


def cone_overflows(levels):
    return max(levels[:-1], default=0) > CONE_CAP or levels[-1] > CONE_HASH


def batch(cx, B1, last, rs, density=0.3):
    """Flows {-1, 0, 1} over the whole complex (every stale cone bit would meet a live row), targets below n_nbrs, a mask with a zero."""
    import scone_gcn_b200 as sg
    last = np.asarray(last, np.int64)
    flows = rs.choice([-1.0, 0.0, 1.0], size=(len(last), cx.E), p=[density / 2, 1 - density, density / 2])[:, :, None]
    _, n_nbrs, _ = so.neighbourhood_tables(B1, last)
    tgt = np.array([rs.randint(0, k) for k in n_nbrs])
    targets = np.zeros((len(last), cx.D, 1))
    targets[np.arange(len(last)), tgt, 0] = 1.0
    mask = np.ones(len(last), np.float32)
    mask[1] = 0.0
    return dict(last=last, flows=flows, targets=targets, tgt=tgt, mask=mask, n_nbrs=n_nbrs, csr=sg.flows_to_csr(flows))


@pytest.fixture(scope='module')
def fan():
    """fan_hub(128, 16) (E = 4096, D = 128) with a batch that overflows the cone kernel (every trajectory ends at the hub) and one that
    fits (rim nodes and leaves), both asserted on the CPU; weights scaled to the fitting batch."""
    import scone_gcn_b200 as sg
    n, edges, faces = fan_hub(128, 16)
    cx = sg.SimplicialComplex.from_simplices(n, edges, faces, 'scone')
    assert (cx.E, cx.D) == (4096, 128)
    B1, B2 = so.incidence_matrices(n, edges, faces)
    L = len(FAN_HIDDEN)
    hub = cone_levels(cx, L, 0)
    assert hub[0] == 128 * 17 > CONE_CAP, hub                                     # the top level is listed: beyond 2048
    rs = np.random.RandomState(31)
    over = batch(cx, B1, [0, 0, 0, 0], rs)
    fit_last = [1, 64, 128, 129, 129 + 8 * 16 + 7, n - 1, 77, 129 + 50 * 16]
    for v in fit_last:
        lv = cone_levels(cx, L, v)
        assert not cone_overflows(lv), (v, lv)
    fit = batch(cx, B1, fit_last, rs)
    fit.update(B1=B1, B2=B2)
    S = [sp.csr_matrix(M) for M in so.shift_matrices(sp.csr_matrix(B1), sp.csr_matrix(B2), 'scone')]
    W, peaks = scaled_weights('scone', B1, S, fit['flows'][:, :, 0], fit['last'], FAN_HIDDEN, rs)
    assert all(1.0 <= q <= 4.0 for q in peaks), peaks
    return dict(cx=cx, over=over, fit=fit, W=W)


def cone_net(fan):
    import scone_gcn_b200 as sg
    net = sg.SconeModel(fan['cx'], FAN_HIDDEN, micro_batch=4)
    net.set_pipeline(3)
    net.set_weights(fan['W'])
    return net


HASH_HIDDEN = [16, 16, 16]


@pytest.fixture(scope='module')
def hubs_batch():
    """The test_gpu_high_degree batch on hubs_8x120; a dense trajectory has a live layer of more merged-row entries than the hash plan's
    slot buffer can hold whatever its size (asserted on the CPU: cone & support, rows of I + S0 + S1)."""
    p = problem('hubs_8x120', 'scone', len(HASH_HIDDEN), seed=5)
    cx = p['cx']
    pat = row_pattern(cx)
    rowlen = np.diff(pat.indptr)
    en = cx._edge_nodes
    nb = cx.nbrhoods[p['last'][0]]
    cone = np.isin(en[:, 0], nb[nb >= 0]) | np.isin(en[:, 1], nb[nb >= 0])
    for _ in range(len(HASH_HIDDEN) - 1):
        cone = (pat @ cone.astype(np.int32)) > 0
    live = cone & ((pat @ (p['flows'][0, :, 0] != 0).astype(np.int32)) > 0)     # live rows of layer 1
    assert int(rowlen[live].sum()) > HASH_SLOTS_MAX, int(rowlen[live].sum())
    rs = np.random.RandomState(2)
    W = [(0.1 * rs.randn(*s)).astype(np.float32) for s in [(1, 16)] * 3 + [(16, 16)] * 6 + [(16, 1)]]
    return p, W


class Dev:
    """A batch as device tensors for the *_dev entry points."""

    def __init__(self, p, D):
        ptr, fe, fv = p['csr']
        t = lambda a, dt: torch.as_tensor(np.ascontiguousarray(a, dt)).cuda()
        self.B = len(p['last'])
        self.ptr, self.fe, self.fv = t(ptr, np.int32), t(fe, np.int32), t(fv, np.float32)
        self.last, self.tgt, self.mask = t(p['last'], np.int32), t(p['tgt'], np.int32), t(p['mask'], np.float32)
        self.lp = torch.zeros(self.B, D, device='cuda')

    def args(self):
        return [C.c_void_p(x.data_ptr()) for x in (self.ptr, self.fe, self.fv, self.last)]

    def loss_grad(self, net):
        import scone_gcn_b200 as sg
        tm = [C.c_void_p(x.data_ptr()) for x in (self.tgt, self.mask)]
        return sg.lib().scone_model_loss_grad_dev(net.handle, self.B, *self.args(), *tm, 1, None)

    def forward(self, net):
        import scone_gcn_b200 as sg
        return sg.lib().scone_model_forward_dev(net.handle, self.B, *self.args(), C.c_void_p(self.lp.data_ptr()), None)


def overflowed(trigger, fan, hubs_batch, monkeypatch):
    """(model with the overflow flag set by a loss_grad_dev that returned 0, batch that fits on the pipeline the model is left on)."""
    if trigger == 'cone':
        net = cone_net(fan)
        over, follow = fan['over'], fan['fit']
    else:
        p, W = hubs_batch
        net = fused_net(monkeypatch, p, HASH_HIDDEN, W, 'hash', 7)
        over = follow = p
    assert Dev(over, net.cx.D).loss_grad(net) == 0
    torch.cuda.synchronize()
    if trigger == 'hash':
        net.set_pipeline(2)                         # the flag belongs to the model: pipeline 2 runs this batch without overflowing
    return net, follow


TRIGGERS = ['cone', 'hash']


@pytest.mark.parametrize('trigger', TRIGGERS)
def test_overflow_triggers_are_deterministic(trigger, fan, hubs_batch, monkeypatch):
    """Each trigger reports code 4 through read_grads, and the batch that follows it does not."""
    net, follow = overflowed(trigger, fan, hubs_batch, monkeypatch)
    with pytest.raises(SconeError, match=r'\(code 4\): scone_model_read_grads:'):
        net.read_grads()
    ptr, fe, fv = follow['csr']
    net.loss_grad(ptr, fe, fv, follow['last'], follow['tgt'], follow['mask'])


@pytest.mark.parametrize('trigger', TRIGGERS)
def test_adam_steps_skip_while_the_flag_is_set(trigger, fan, hubs_batch, monkeypatch):
    """After an overflowing loss_grad_dev: two adam_steps and a one-rank exchange step leave W bit-identical (the exchange still writes
    the buffer back); once the flag is reported and cleared, the next step is the float64 reference's from the moments of before."""
    import scone_gcn_b200 as sg
    net, _ = overflowed(trigger, fan, hubs_batch, monkeypatch)
    n = net.n_params
    rs = np.random.RandomState(4)
    wd = 5e-5
    # a clean step first, so that the moments are not zero: the flag of the first trigger is reported (and cleared) ...
    with pytest.raises(SconeError, match=r'\(code 4\)'):
        net.check_overflow()
    W0 = weights(net)
    buf0 = chosen_buffer(n, 37.0, rs)
    write_buffer(net, buf0)
    net.adam_step(0, LR, wd)
    W1 = weights(net)
    W_ref, m, v = adam64(0, buf0, W0, np.zeros(n), np.zeros(n), LR, wd)
    check_step(W1, W0, W_ref, 0, LR, 'set-up')
    # ... and the same model overflows again (the cone model stays on pipeline 3; the hash model goes back to its fused pipeline)
    if trigger == 'cone':
        assert Dev(fan['over'], net.cx.D).loss_grad(net) == 0
    else:
        net.set_pipeline(4)
        assert Dev(hubs_batch[0], net.cx.D).loss_grad(net) == 0
    for i in (1, 2):
        net.adam_step(i, LR, wd)
        assert np.array_equal(weights(net).view(np.uint32), W1.view(np.uint32)), ('adam_step', i)
    negz = np.arange(1, n, 9)
    buf = chosen_buffer(n, 12.0, rs, neg_zeros=negz)
    write_buffer(net, buf)
    rc, dp = dp_create(n + 2)
    assert rc == 0
    try:
        assert dp_step(net, dp, 1, LR, wd) == 0
        assert sg.lib().scone_dp_status(dp, None) == 0
    finally:
        sg.lib().scone_dp_destroy(dp)
    assert np.array_equal(weights(net).view(np.uint32), W1.view(np.uint32)), 'exchange step'
    back = device_buffer(net)
    assert np.array_equal(back, buf) and not np.signbit(back[negz]).any()              # written back (0 + x) although skipped
    with pytest.raises(SconeError, match=r'\(code 4\): scone_model_check_overflow:'):
        net.check_overflow()
    net.adam_step(1, LR, wd)
    got = weights(net)
    W_ref, _, _ = adam64(1, back, W1, m, v, LR, wd)
    print('adam after overflow (%s): worst err/tol %.3g' % (trigger, check_step(got, W1, W_ref, 1, LR, 'after the overflow')))


ENTRY_POINTS = ['check_overflow', 'read_grads', 'forward_host', 'accuracy_host', 'eval_host']


def call_entry(net, name, p):
    ptr, fe, fv = p['csr']
    if name == 'check_overflow':
        net.check_overflow()
    elif name == 'read_grads':
        net.read_grads()
    elif name == 'forward_host':
        net.forward(ptr, fe, fv, p['last'])
    elif name == 'accuracy_host':
        net.accuracy(ptr, fe, fv, p['last'], p['n_nbrs'], p['tgt'], p['mask'])
    else:
        net.evaluate(ptr, fe, fv, p['last'], n_nbrs=p['n_nbrs'], target_idx=p['tgt'], mask=p['mask'], want_choice=True,
                     want_accuracy=True, want_nll=True)


@pytest.mark.parametrize('entry', ENTRY_POINTS)
@pytest.mark.parametrize('trigger', TRIGGERS)
def test_overflow_is_reported_once_by_each_reporting_entry_point(trigger, entry, fan, hubs_batch, monkeypatch):
    """While the flag is set, loss_grad_dev, forward_dev, read_grads_async and adam_step return 0; then `entry` returns 4 naming
    itself, and the very next call returns 0.  After an eval_host that reported 4, two_target_host is refused (code 2)."""
    net, follow = overflowed(trigger, fan, hubs_batch, monkeypatch)
    d = Dev(follow, net.cx.D)
    assert d.forward(net) == 0 and d.loss_grad(net) == 0
    pinned = torch.empty(net.n_params + 2, dtype=torch.float32, pin_memory=True)
    net.read_grads_async(pinned)
    W = weights(net)
    net.adam_step(0, LR, 5e-5)
    torch.cuda.synchronize()
    assert np.array_equal(weights(net).view(np.uint32), W.view(np.uint32))
    rnd = (follow['tgt'] + 1) % np.maximum(follow['n_nbrs'], 1)
    with pytest.raises(SconeError, match=r'\(code 4\): scone_model_%s:' % entry):
        call_entry(net, entry, follow)
    if entry == 'eval_host':
        with pytest.raises(SconeError, match=r'\(code 2\): scone_model_two_target_host:'):
            net.two_target_counts(follow['tgt'], rnd)
    call_entry(net, entry, follow)
    net.check_overflow()
    if entry == 'eval_host':
        net.two_target_counts(follow['tgt'], rnd)


@pytest.fixture(scope='module')
def fan_fresh(fan):
    """A fresh model's log-probs and gradient buffer of the fitting batch on pipeline 3, checked against the float64 oracle."""
    fit = fan['fit']
    ref = Oracle(dict(fit, cx=fan['cx']), 'scone', fan['W'])
    net = cone_net(fan)
    return check_vs_oracle(net, fit, ref, 'fresh, pipeline 3')


@pytest.mark.parametrize('variant', ['once', 'fitting batch twice', 'two overflows'])
def test_cone_pipeline_recovers_after_a_reported_overflow(variant, fan, fan_fresh):
    """Overflowing batch (reported), then the fitting batch on the same pipeline-3 model: log-probs and gradient buffer bit-identical to
    a fresh model's (which match the float64 oracle).  A truncated cone list may leave bitmap bits the per-batch clearing misses; the
    report makes the next batch clear every bitmap."""
    net = cone_net(fan)
    over, fit = fan['over'], fan['fit']
    for _ in range(2 if variant == 'two overflows' else 1):
        ptr, fe, fv = over['csr']
        with pytest.raises(SconeError, match=r'\(code 4\): scone_model_read_grads:'):
            net.loss_grad(ptr, fe, fv, over['last'], over['tgt'], over['mask'])
    lp0, buf0 = fan_fresh
    ptr, fe, fv = fit['csr']
    for _ in range(2 if variant == 'fitting batch twice' else 1):
        lp = net.forward(ptr, fe, fv, fit['last'])
        buf = net.loss_grad(ptr, fe, fv, fit['last'], fit['tgt'], fit['mask'])
        assert np.array_equal(lp.view(np.uint32), lp0.view(np.uint32)), variant
        assert np.array_equal(buf.view(np.uint32), buf0.view(np.uint32)), (variant, np.flatnonzero(buf != buf0)[:8])

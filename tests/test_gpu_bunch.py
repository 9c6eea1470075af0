"""-model bunch (SCCONV) against a float64 reference at every layer-width path, depth, micro-batch split and complex shape.

Paths of csrc/scone_bunch.cu and the hidden lists that reach them:
  fused level kernels (widths 1 / 8 / 16)   [16,16,16] (the cfg3-bunch bench shape), [8,16], [16,8], [1], [1,1], [8], [8,8,8,8,8]
  generic kernels (any other width)         [32,32] (16 weight-gradient tiles: kOuterTilesMax), [40,40] / [64,64] (outer_reduce_kernel),
                                            [3], [5,5] (odd widths, masked partial tiles)
  fused <-> generic boundaries              [12,8], [8,12,16]
on the hand-built complexes (a path without triangles: F = 0, isolated nodes, leaves, D up to 200) and on the reference's datasets.

The reference is oracle.DenseOracle('bunch') in float64 where dense products are cheap (max(E, F) <= DENSE_MAX_ROWS), and SparseBunchRef below
(the same recurrence over torch.sparse float64 operators, checked against DenseOracle to 1e-12) on dataset_default and the hub complexes.
Weights are drawn per layer and rescaled so the float64 pre-activations are not degenerate (20-80 % of the non-zero ones positive,
logits peaking at 2.5): a batch of dead ReLUs cannot pass by producing zeros on both sides."""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

from golden_util import Dataset
from oracle import scone_oracle as so
from scone_gcn_b200.bunch_model_matrices import compute_shift_matrices
from test_index_tiny_complexes import CASES, wheel

DENSE_MAX_ROWS = 300                 # DenseOracle when max(E, F) is at most this, SparseBunchRef above
PEAK_LOGIT = 2.5
POSITIVE_SHARE = (0.2, 0.8)          # share of positive pre-activations among the non-zero ones, per layer
COMPLEXES = dict(CASES, wheel_200=wheel(200))    # wheel_200 (D = 200) is beyond the scone model's degree limit, not the bunch model's
OUT_LEVEL = (0, 0, 1, 1, 1, 2, 2)    # level (0 nodes, 1 edges, 2 triangles) term k writes: S_00, S_10, S_01, S_11, S_21, S_12, S_22
IN_LEVEL = (0, 1, 0, 1, 2, 1, 2)     # level term k reads


def structurally_zero(layer, k, L, F):
    """Weights whose gradient is exactly zero whatever the data: layer 0 reads V_0 = T_0 = 0 (S_00, S_01, S_21, S_22); the readout
    reads only the nodes of the last layer, so its edge and triangle outputs, and the triangles of the layer before (read only by
    the last layer's edge and triangle terms), reach no loss; with F = 0, S_21, S_12 and S_22 are empty."""
    return ((layer == 0 and IN_LEVEL[k] != 1) or (layer == L - 1 and OUT_LEVEL[k] != 0) or (layer == L - 2 and OUT_LEVEL[k] == 2)
            or (F == 0 and 2 in (IN_LEVEL[k], OUT_LEVEL[k])))


class SparseBunchRef:
    """bunch_func (trajectory_experiments.py:173-203) over torch.sparse float64 operators, autograd for the gradients.

    States are [rows, B, C].  Everything else is DenseOracle('bunch'): its activation (torch.maximum, ties split), V_0 = T_0 = 0 and
    X = the flows, relu after every layer, the -1 -> node N-1 wrap of padded slots (Q2), log-softmax over all D slots and the loss
    -sum(mask * logp[target]) / sum(mask) + wd * sum(w^2)."""

    def __init__(self, shifts, nbrhoods, device='cpu'):
        self.dev = torch.device(device)
        self.S = []
        for M in shifts:
            M = sp.coo_matrix(M)
            idx = torch.as_tensor(np.vstack([M.row, M.col]).astype(np.int64))
            self.S.append(torch.sparse_coo_tensor(idx, torch.as_tensor(M.data, dtype=torch.float64), M.shape).coalesce().to(self.dev))
        self.N, self.E, self.F = shifts[0].shape[0], shifts[3].shape[0], shifts[6].shape[0]
        self.nbr = torch.as_tensor(np.asarray(nbrhoods, np.int64), device=self.dev)
        self.act = so._ACT['bunch']

    def _shift(self, k, X):
        rows, (cols, B, C) = self.S[k].shape[0], X.shape
        if rows == 0 or cols == 0:
            return X.new_zeros(rows, B, C)
        return torch.sparse.mm(self.S[k], X.reshape(cols, B * C)).reshape(rows, B, C)

    def inputs(self, flows):
        X = torch.as_tensor(np.asarray(flows, np.float64).reshape(len(flows), -1).T.copy(), device=self.dev)     # [E, B]
        B = X.shape[1]
        return [X.new_zeros(self.N, B, 1), X.reshape(self.E, B, 1), X.new_zeros(self.F, B, 1)]

    def layer(self, cur, W):
        """Pre-activations (nodes, edges, triangles) of one layer; W = its 7 weights (trajectory_experiments.py:184-192)."""
        t = lambda k, lv: self._shift(k, cur[lv]) @ W[k]
        return [t(0, 0) + t(1, 1), t(2, 0) + t(3, 1) + t(4, 2), t(5, 1) + t(6, 2)]

    def logits(self, V, last_nodes):
        Nv = self.nbr[torch.as_tensor(np.asarray(last_nodes, np.int64), device=self.dev)] % self.N      # [B, D]; -1 -> N - 1
        return torch.gather(V[:, :, 0].T, 1, Nv)

    def weights(self, W):
        return [w if isinstance(w, torch.Tensor) else torch.as_tensor(np.asarray(w, np.float64), device=self.dev) for w in W]

    def forward(self, W, flows, last_nodes, pre=None):
        """log-probs [B, D]; the pre-activations of every layer are appended to `pre` when it is given."""
        W = self.weights(W)
        cur = self.inputs(flows)
        for i in range(len(W) // 7):
            z = self.layer(cur, W[7 * i:7 * i + 7])
            if pre is not None:
                pre.append(z)
            cur = [self.act(x) for x in z]
        lg = self.logits(cur[0], last_nodes)
        return lg - torch.logsumexp(lg, dim=1, keepdim=True)

    def loss_and_grads(self, W, flows, last_nodes, target_idx, mask, wd=0.0):
        """(mean loss, masked nll sum, [dW] as numpy) — DenseOracle.loss_and_grads with the nll sum the library accumulates."""
        W = [w.clone().requires_grad_(True) for w in self.weights(W)]
        lp = self.forward(W, flows, last_nodes)
        m = torch.as_tensor(np.asarray(mask) == 1, device=self.dev)
        tgt = torch.as_tensor(np.asarray(target_idx, np.int64), device=self.dev)
        nll = -lp[torch.arange(len(tgt), device=self.dev), tgt][m].sum()
        loss = nll / m.sum() + wd * sum((w ** 2).sum() for w in W)
        g = torch.autograd.grad(loss, W)
        return float(loss.detach()), float(nll.detach()), [x.detach().cpu().numpy() for x in g]


def nonzero_positive_share(z):
    v = torch.cat([x.reshape(-1) for x in z])
    v = v[v != 0]
    return float((v > 0).double().mean()) if len(v) else 0.0


def levels_alive(z):
    """Each level with at least 10 non-zero pre-activations has 10-90 % of them positive (a width-1 layer can otherwise lose its whole
    node level while the edge level keeps the layer's share in range)."""
    for x in z:
        v = x[x != 0]
        if len(v) >= 10 and not 0.1 <= float((v > 0).double().mean()) <= 0.9:
            return False
    return True


def calibrated_weights(ref, hidden, flows, last_nodes, seed):
    """fp32 weights, layer by layer: 7 standard-normal arrays, redrawn until 25-75 % of the layer's non-zero fp64 pre-activations are
    positive (and no level is all but dead), then scaled (relu is positively homogeneous: the share does not move) so the largest |pre-activation| of a hidden layer
    is 1 and the largest logit is PEAK_LOGIT."""
    rs = np.random.RandomState(seed)
    widths = [1] + list(hidden) + [1]
    cur = ref.inputs(flows)
    W = []
    for i in range(len(widths) - 1):
        last_layer = i == len(widths) - 2
        for _ in range(50):
            Wi = [rs.randn(widths[i], widths[i + 1]) for _ in range(7)]
            z = ref.layer(cur, ref.weights(Wi))
            share = nonzero_positive_share(z)
            top = float(ref.logits(ref.act(z[0]), last_nodes).max()) if last_layer else max(float(x.abs().max()) for x in z if x.numel())
            if 0.25 <= share <= 0.75 and levels_alive(z) and top > 0:
                break
        else:
            raise AssertionError('no non-degenerate draw for layer %d' % i)
        s = (PEAK_LOGIT if last_layer else 1.0) / top
        Wi = [(w * s).astype(np.float32) for w in Wi]
        W += Wi
        cur = [ref.act(x) for x in ref.layer(cur, ref.weights(Wi))]
    return W


def assert_not_degenerate(ref, W, flows, last_nodes):
    pre = []
    with torch.no_grad():
        ref.forward(W, flows, last_nodes, pre)
    for i, z in enumerate(pre):
        share = nonzero_positive_share(z)
        assert POSITIVE_SHARE[0] <= share <= POSITIVE_SHARE[1], (i, share)
    peak = float(ref.logits(ref.act(pre[-1][0]), last_nodes).max())
    assert 2.0 <= peak <= 3.0, peak


# ---- problems ----------------------------------------------------------------------------------------------------------------------
class Problem:
    """A complex, its seven operators, neighbour table and a batch of trajectories (flows [B, E, 1], last nodes, targets, mask)."""

    def __init__(self, B1, B2, flows, last_nodes, tgt, mask):
        self.B1, self.B2 = B1, B2
        self.shifts = compute_shift_matrices(B1, B2)
        self.nbrhoods = so.neighbourhood_tables(B1, last_nodes)[0]
        self.N, self.D = self.nbrhoods.shape
        self.E, self.F = B1.shape[1], B2.shape[1]
        self.flows, self.last_nodes, self.tgt = flows, np.asarray(last_nodes), np.asarray(tgt)
        self.mask = np.asarray(mask, np.float32)
        self.B = len(self.last_nodes)

    def csr(self):
        import scone_gcn_b200 as sg
        return sg.flows_to_csr(self.flows)

    def ops(self):
        from scone_gcn_b200.bunch import CsrOperator
        return [CsrOperator(M) for M in self.shifts]

    def model(self, hidden, micro_batch):
        from scone_gcn_b200.bunch import BunchModel
        return BunchModel(self.ops(), self.nbrhoods, hidden, micro_batch=micro_batch)

    def subset(self, idx):
        p = Problem.__new__(Problem)
        p.__dict__.update(self.__dict__)
        p.flows, p.last_nodes, p.tgt, p.mask = self.flows[idx], self.last_nodes[idx], self.tgt[idx], self.mask[idx]
        p.B = len(p.last_nodes)
        return p


def complex_problem(name, seed=0):
    """As test_gpu_tiny_complexes.tiny_problem: one trajectory ending at every node (isolated ones included), trajectory 0 empty
    (all logits 0), a random target among each last node's neighbours, trajectory 1 masked out; flows of either sign on 60 % of
    the edges."""
    n, edges, faces = COMPLEXES[name]
    edges, faces = np.asarray(edges, np.int64).reshape(-1, 2), np.asarray(faces, np.int64).reshape(-1, 3)
    B1, B2 = so.incidence_matrices(n, edges, faces)
    rs = np.random.RandomState(seed)
    flows = rs.choice([-1.0, 0.0, 1.0], size=(n, len(edges), 1), p=[0.3, 0.4, 0.3])
    # magnitudes in [0.5, 1.5): with unit flows the regular operators of these complexes cancel exactly at many rows, which puts those
    # pre-activations on the ReLU kink in exact arithmetic, and fp32 and fp64 rounding then pick different sides of it
    flows = (flows * rs.uniform(0.5, 1.5, size=flows.shape)).astype(np.float32).astype(np.float64)
    flows[0] = 0.0
    last_nodes = np.arange(n)
    _, n_nbrs, _ = so.neighbourhood_tables(B1, last_nodes)
    tgt = np.array([rs.randint(0, max(1, k)) for k in n_nbrs])
    mask = np.ones(n)
    mask[1] = 0.0
    return Problem(B1, B2, flows, last_nodes, tgt, mask)


_DATASETS = {}


def dataset_problem(which):
    if which not in _DATASETS:
        ds = Dataset('dataset_%s.npz' % which)
        _DATASETS[which] = Problem(ds.B1, ds.B2, ds.flows, ds.last_nodes, ds.raw['targets_argmax'], ds.train_mask)
    return _DATASETS[which]


def reference(p, W, device):
    """(log-probs [B, D], masked nll sum, [dW] of the mean loss) in float64."""
    if max(p.E, p.F) <= DENSE_MAX_ROWS:
        targets = np.zeros((p.B, p.D, 1))
        targets[np.arange(p.B), p.tgt, 0] = 1.0
        orc = so.DenseOracle('bunch', [M.toarray() for M in p.shifts], p.B1, p.last_nodes, p.flows, targets, dtype=torch.float64)
        with torch.no_grad():
            lp = orc.forward(W).numpy()[:, :, 0]
        loss, g = orc.loss_and_grads(W, p.mask, 0.0)
        return lp, float(loss) * float((p.mask == 1).sum()), g
    ref = SparseBunchRef(p.shifts, p.nbrhoods, device)
    with torch.no_grad():
        lp = ref.forward(W, p.flows, p.last_nodes).cpu().numpy()
    _, nll, g = ref.loss_and_grads(W, p.flows, p.last_nodes, p.tgt, p.mask)
    return lp, nll, g


def grad_err(grads, g_ref):
    """Largest error of any array relative to its bound: <= 1 passes.  Per array, relative to its largest entry; an array whose true
    gradient is zero up to fp32 cancellation noise is held to the noise floor instead (the rule of test_gpu_tiny_complexes.py)."""
    gmax = max(float(np.abs(r).max()) for r in g_ref if r.size)
    return max(float(np.abs(a - r).max()) / (1e-4 * max(float(np.abs(r).max()), 1e-3 * gmax, 1e-2)) for a, r in zip(grads, g_ref))


def check_against_reference(p, hidden, micro_batch, seed=1, tag=''):
    """Forward and loss_grad of a fresh BunchModel against the float64 reference; returns (model, weights, grad buffer)."""
    import scone_gcn_b200 as sg  # noqa: F401
    dev = 'cuda' if torch.cuda.is_available() else 'cpu'
    ref = SparseBunchRef(p.shifts, p.nbrhoods, dev)
    L = len(hidden) + 1
    for seed in range(seed, seed + 10):
        # a narrow layer can still route all of one weight's signal away from the readout (width 1: the node level lights up only
        # around the first node of each trajectory): redraw until every array that can have a gradient has one
        W = calibrated_weights(ref, hidden, p.flows, p.last_nodes, seed)
        lp_ref, nll_ref, g_ref = reference(p, W, dev)
        if all(np.any(r != 0.0) for i, r in enumerate(g_ref) if not structurally_zero(*divmod(i, 7), L, p.F)):
            break
    assert_not_degenerate(ref, W, p.flows, p.last_nodes)
    net = p.model(hidden, micro_batch)
    net.set_weights(W)
    ptr, fe, fv = p.csr()
    lp = net.forward(ptr, fe, fv, p.last_nodes)
    lp_err = float(np.abs(lp - lp_ref).max())
    assert lp_err <= 1e-5 * max(1.0, float(np.abs(lp_ref).max())), lp_err
    buf = net.loss_grad(ptr, fe, fv, p.last_nodes, p.tgt, p.mask)
    n = net.n_params
    assert buf[n + 1] == p.mask.sum()
    assert buf[n] == pytest.approx(nll_ref, rel=1e-5)
    grads = net.unflatten(buf[:n] / buf[n + 1])
    gerr = grad_err(grads, g_ref)
    print('[bunch-err] %-32s hidden=%-16s mb=%-5d |dlogp| %.2e  grad err %.3f of the bound' % (tag, hidden, micro_batch, lp_err, gerr))
    assert gerr <= 1.0, gerr
    assert len(grads) == 7 * L
    for i, (a, r) in enumerate(zip(grads, g_ref)):
        layer, k = divmod(i, 7)
        if structurally_zero(layer, k, L, p.F):
            assert np.all(a == 0.0) and np.all(r == 0.0), (layer, k)
        else:
            assert np.any(r != 0.0) and np.any(a != 0.0), (layer, k)
    return net, W, buf


# ---- the float64 references agree ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('name', ['dataset_small', 'path_without_triangles', 'star_max_degree_and_leaves'])
def test_sparse_reference_matches_dense_oracle(name):
    p = dataset_problem('small') if name == 'dataset_small' else complex_problem(name)
    ref = SparseBunchRef(p.shifts, p.nbrhoods)
    W = calibrated_weights(ref, [8, 5], p.flows, p.last_nodes, seed=3)
    wd = 1e-2
    targets = np.zeros((p.B, p.D, 1))
    targets[np.arange(p.B), p.tgt, 0] = 1.0
    orc = so.DenseOracle('bunch', [M.toarray() for M in p.shifts], p.B1, p.last_nodes, p.flows, targets, dtype=torch.float64)
    with torch.no_grad():
        lp_d = orc.forward(W).numpy()[:, :, 0]
        lp_s = ref.forward(W, p.flows, p.last_nodes).numpy()
    assert np.abs(lp_s - lp_d).max() <= 1e-12 * max(1.0, np.abs(lp_d).max())
    loss_d, g_d = orc.loss_and_grads(W, p.mask, wd)
    loss_s, _, g_s = ref.loss_and_grads(W, p.flows, p.last_nodes, p.tgt, p.mask, wd)
    assert abs(loss_s - float(loss_d)) <= 1e-12 * max(1.0, abs(float(loss_d)))
    gmax = max(np.abs(g).max() for g in g_d)
    assert gmax > 0
    for a, r in zip(g_s, g_d):
        assert np.abs(a - r).max() <= 1e-12 * max(1.0, gmax)


# ---- widths and depths on dataset_small --------------------------------------------------------------------------------------------
HIDDEN = [
    [16, 16, 16],               # the cfg3-bunch bench shape: fused (1,16), (16,16), (16,1)
    [8, 16], [16, 8],           # mixed fused widths
    [1], [1, 1],                # fused (1,1)
    [32, 32],                   # generic; 4 x 4 = 16 weight-gradient tiles, exactly kOuterTilesMax
    [40, 40], [64, 64],         # generic; 25 / 64 tiles: outer_reduce_kernel
    [12, 8], [8, 12, 16],       # fused -> generic -> fused boundaries; masked partial tiles
    [3], [5, 5],                # odd widths
    [8],                        # one hidden layer
    [8, 8, 8, 8, 8],            # five hidden layers
]


@pytest.mark.gpu
@pytest.mark.parametrize('hidden', HIDDEN, ids=lambda h: 'h' + '_'.join(map(str, h)))
def test_widths_and_depths_vs_reference(hidden):
    check_against_reference(dataset_problem('small'), hidden, micro_batch=32, tag='dataset_small')


# ---- complex shapes -----------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('hidden', [[8, 8], [16, 16]], ids=lambda h: 'h' + '_'.join(map(str, h)))
@pytest.mark.parametrize('name', sorted(COMPLEXES))
def test_complexes_vs_reference(name, hidden):
    p = complex_problem(name)
    if name == 'path_without_triangles':
        assert p.F == 0 and [M.shape for M in p.shifts][4:] == [(4, 0), (0, 4), (0, 0)]
    if name == 'wheel_200':
        assert p.D == 200
    check_against_reference(p, hidden, micro_batch=32, tag=name)


@pytest.mark.gpu
def test_zero_size_operators_are_accepted():
    from scone_gcn_b200.bunch import CsrOperator
    for shape in [(4, 0), (0, 4), (0, 0)]:
        S = CsrOperator(sp.csr_matrix(shape))
        assert S.shape == shape and S.handle


# ---- the bench shape ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('micro_batch', [1000, 300])
def test_bench_shape_on_dataset_default(micro_batch):
    """bench_bunch's configuration: hidden 16-16-16 over all 1000 trajectories (micro-batch min(B, 1024)); 300 leaves a tail of 100."""
    p = dataset_problem('default')
    assert p.B == 1000
    check_against_reference(p, [16, 16, 16], micro_batch, tag='dataset_default')


# ---- micro-batch split and determinism ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('hidden', [[16, 16, 16], [12, 8]], ids=lambda h: 'h' + '_'.join(map(str, h)))
def test_micro_batch_split_and_determinism(hidden):
    p = dataset_problem('small')
    ref = SparseBunchRef(p.shifts, p.nbrhoods)
    W = calibrated_weights(ref, hidden, p.flows, p.last_nodes, seed=5)
    ptr, fe, fv = p.csr()
    lps, bufs = {}, {}
    for mb in (1, 7, p.B, p.B + 5):
        net = p.model(hidden, mb)
        net.set_weights(W)
        lps[mb] = net.forward(ptr, fe, fv, p.last_nodes)
        bufs[mb] = net.loss_grad(ptr, fe, fv, p.last_nodes, p.tgt, p.mask)
        again = net.loss_grad(ptr, fe, fv, p.last_nodes, p.tgt, p.mask)
        assert np.array_equal(bufs[mb], again), mb                    # same micro-batch: bit-identical gradients
    n = net.n_params
    for mb in lps:
        # every (row, trajectory) value of the forward is computed independently of the micro-batch
        assert np.array_equal(lps[mb], lps[1]), mb
        assert bufs[mb][n + 1] == p.mask.sum()
        assert bufs[mb][n] == pytest.approx(bufs[p.B][n], rel=1e-5)
        g = net.unflatten(bufs[mb][:n] / bufs[mb][n + 1])
        g_full = net.unflatten(bufs[p.B][:n] / bufs[p.B][n + 1])
        assert grad_err(g, g_full) <= 1.0, mb


# ---- host contract -----------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_accumulation_across_calls_equals_one_call():
    p = dataset_problem('small')
    net, W, full = check_against_reference(p, [16, 16], micro_batch=16, tag='accumulate')
    ptr_a, fe_a, fv_a = sg_csr(p.flows[:23])
    ptr_b, fe_b, fv_b = sg_csr(p.flows[23:])
    net.loss_grad(ptr_a, fe_a, fv_a, p.last_nodes[:23], p.tgt[:23], p.mask[:23], zero_first=True, read=False)
    two = net.loss_grad(ptr_b, fe_b, fv_b, p.last_nodes[23:], p.tgt[23:], p.mask[23:], zero_first=False)
    n = net.n_params
    assert two[n + 1] == full[n + 1] == p.mask.sum()
    assert two[n] == pytest.approx(full[n], rel=1e-5)
    assert grad_err(net.unflatten(two[:n]), net.unflatten(full[:n])) <= 1.0


def sg_csr(flows):
    import scone_gcn_b200 as sg
    return sg.flows_to_csr(flows)


@pytest.mark.gpu
def test_empty_batch_calls():
    import scone_gcn_b200 as sg
    p = dataset_problem('small')
    net = p.model([8, 8], 16)                    # fresh: nothing staged yet
    ref = SparseBunchRef(p.shifts, p.nbrhoods)
    net.set_weights(calibrated_weights(ref, [8, 8], p.flows, p.last_nodes, seed=2))
    empty = (np.zeros(1, np.int32), np.zeros(0, np.int32), np.zeros(0, np.float32))
    none_i, none_f = np.zeros(0, np.int32), np.zeros(0, np.float32)
    n0 = sg.lib().scone_launch_count()
    assert net.forward(*empty, none_i).shape == (0, p.D)
    assert np.all(net.loss_grad(*empty, none_i, none_i, none_f, zero_first=True) == 0.0)
    assert sg.lib().scone_launch_count() == n0
    ptr, fe, fv = p.csr()
    before = net.loss_grad(ptr, fe, fv, p.last_nodes, p.tgt, p.mask)
    assert before[net.n_params + 1] == p.mask.sum()
    n0 = sg.lib().scone_launch_count()
    assert np.array_equal(net.loss_grad(*empty, none_i, none_i, none_f, zero_first=False), before)      # left as it is
    assert np.all(net.loss_grad(*empty, none_i, none_i, none_f, zero_first=True) == 0.0)                # cleared
    assert sg.lib().scone_launch_count() == n0


def adam_reference(i, grad_buf, W, state, lr, wd):
    """oracle.adam_update in fp32 on the kernel's own gradient buffer: g = grads / count + 2 wd W (scone_adam_launch)."""
    n = grad_buf.size - 2
    g = grad_buf[:n] / grad_buf[n + 1] + np.float32(2 * wd) * W
    (x, m, v), = so.adam_update(i, [g.astype(np.float32)], [(W, state[0], state[1])], lr, dtype=np.float32)
    return x, (m, v)


@pytest.mark.gpu
def test_adam_steps_match_oracle_update():
    p = dataset_problem('small')
    net, W, _ = check_against_reference(p, [16, 16], micro_batch=32, tag='adam')
    ptr, fe, fv = p.csr()
    lr, wd = 1e-2, 5e-3
    w = net.flatten(W)
    state = (np.zeros_like(w), np.zeros_like(w))
    for step in range(2):
        buf = net.loss_grad(ptr, fe, fv, p.last_nodes, p.tgt, p.mask)
        net.adam_step(step, lr, wd)
        x, state = adam_reference(step, buf, w, state, lr, wd)
        got = net.flatten(net.get_weights())
        np.testing.assert_allclose(got, x, rtol=1e-6, atol=1e-4 * lr)
        w = got


@pytest.mark.gpu
def test_set_weights_without_reset_keeps_adam_moments():
    p = dataset_problem('small')
    net, W, _ = check_against_reference(p, [8, 12, 16], micro_batch=32, tag='set_weights')
    ptr, fe, fv = p.csr()
    lr, wd = 1e-2, 5e-3
    w0 = net.flatten(W)
    buf = net.loss_grad(ptr, fe, fv, p.last_nodes, p.tgt, p.mask)
    net.adam_step(0, lr, wd)
    _, state = adam_reference(0, buf, w0, (np.zeros_like(w0), np.zeros_like(w0)), lr, wd)
    W2 = [np.float32(0.5) * w for w in W]                          # new weights, same moments
    net.set_weights(W2, reset_adam=False)
    w2 = net.flatten(W2)
    buf = net.loss_grad(ptr, fe, fv, p.last_nodes, p.tgt, p.mask)
    net.adam_step(1, lr, wd)
    got = net.flatten(net.get_weights())
    keep, _ = adam_reference(1, buf, w2, state, lr, wd)
    reset, _ = adam_reference(1, buf, w2, (np.zeros_like(w2), np.zeros_like(w2)), lr, wd)
    np.testing.assert_allclose(got, keep, rtol=1e-6, atol=1e-4 * lr)
    assert np.abs(got - reset).max() > 1e-2 * lr                  # a reset would have given a visibly different step


# ---- rejections --------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_bad_hidden_widths_and_neighbour_tables_are_rejected():
    import scone_gcn_b200 as sg
    from scone_gcn_b200._lib import SconeError
    from scone_gcn_b200.bunch import BunchModel
    p = complex_problem('star_max_degree_and_leaves')
    ops = p.ops()
    n0 = sg.lib().scone_launch_count()
    for hidden, bad in [([8, 0], 0), ([-3], -3)]:
        with pytest.raises(SconeError, match=r'code 2\): .*hidden width %d of layer' % bad):
            BunchModel(ops, p.nbrhoods, hidden)
    for value in (p.N, -2):
        nb = p.nbrhoods.copy()
        nb[3, 1] = value
        with pytest.raises(SconeError, match=r'code 2\): .*nbrhoods\[3\]\[1\] = %d is outside \[-1, %d\)' % (value, p.N)):
            BunchModel(ops, nb, [8])
    assert sg.lib().scone_launch_count() == n0


@pytest.mark.gpu
def test_bad_last_nodes_and_targets_are_rejected():
    import scone_gcn_b200 as sg
    from scone_gcn_b200._lib import SconeError
    p = complex_problem('star_max_degree_and_leaves')
    net = p.model([8], 4)
    ptr, fe, fv = p.csr()
    before = net.loss_grad(ptr, fe, fv, p.last_nodes, p.tgt, p.mask)
    n0 = sg.lib().scone_launch_count()
    for value in (-1, p.N):
        last = p.last_nodes.copy()
        last[2] = value
        with pytest.raises(SconeError, match=r'code 2\): .*last_nodes\[2\] = %d is outside \[0, %d\)' % (value, p.N)):
            net.forward(ptr, fe, fv, last)
        with pytest.raises(SconeError, match=r'code 2\): .*last_nodes\[2\] = %d is outside \[0, %d\)' % (value, p.N)):
            net.loss_grad(ptr, fe, fv, last, p.tgt, p.mask, read=False)
    for value in (-1, p.D):
        tgt = p.tgt.copy()
        tgt[4] = value
        with pytest.raises(SconeError, match=r'code 2\): .*target_idx\[4\] = %d is outside \[0, %d\)' % (value, p.D)):
            net.loss_grad(ptr, fe, fv, p.last_nodes, tgt, p.mask, zero_first=True, read=False)
    assert sg.lib().scone_launch_count() == n0
    assert np.array_equal(net.read_grads(), before)                 # rejected before the buffer was cleared

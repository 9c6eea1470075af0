"""Index construction on hand-built complexes (SURVEY 4 (i)/(ii)): the library's exact integer CSR operators and neighbour table
against the oracle's dense restatement of the reference (`incidence_matrices`, `B1.T @ B1`, `B2 @ B2.T`, `nbrhoods`) — bit-exact,
no GPU needed (`scone_complex_create_index_only`)."""
import itertools

import numpy as np
import pytest

from oracle import scone_oracle as so


def wheel(n_rim):
    """Hub 0, rim 1..n_rim as a cycle, faces (0, i, i + 1): the hub has degree n_rim, every rim node degree 3."""
    rim = list(range(1, n_rim + 1))
    cyc = [tuple(sorted((a, b))) for a, b in zip(rim, rim[1:] + rim[:1])]
    edges = sorted([(0, v) for v in rim] + cyc)
    faces = sorted((0,) + e for e in cyc)
    return n_rim + 1, edges, faces


def hubs(n_hubs, n_rim):
    """Hubs 0..n_hubs-1 pairwise joined and each joined to all rim nodes n_hubs..; faces: every (hub, hub, rim) and (hub, hub, hub).
    A hub has degree n_hubs - 1 + n_rim; its readout touches every edge of the complex."""
    H, R = range(n_hubs), range(n_hubs, n_hubs + n_rim)
    edges = sorted(list(itertools.combinations(H, 2)) + [(h, r) for h in H for r in R])
    faces = sorted([a + (r,) for a in itertools.combinations(H, 2) for r in R] + list(itertools.combinations(H, 3)))
    return n_hubs + n_rim, edges, faces


CASES = {
    # name: (n_nodes, edges (a < b, lexicographic), faces (a < b < c))
    'single_triangle': (3, [(0, 1), (0, 2), (1, 2)], [(0, 1, 2)]),
    'two_triangles_sharing_an_edge': (4, [(0, 1), (0, 2), (1, 2), (1, 3), (2, 3)], [(0, 1, 2), (1, 2, 3)]),
    'path_without_triangles': (5, [(0, 1), (1, 2), (2, 3), (3, 4)], []),
    'isolated_nodes': (6, [(0, 1), (0, 2), (1, 2)], [(0, 1, 2)]),                       # nodes 3, 4, 5 have no edges
    'star_max_degree_and_leaves': (7, [(0, 1), (0, 2), (0, 3), (0, 4), (0, 5), (0, 6), (1, 2)], [(0, 1, 2)]),
    'triangle_fan_with_open_edge': (5, [(0, 1), (0, 2), (0, 3), (0, 4), (1, 2), (2, 3)], [(0, 1, 2), (0, 2, 3)]),
    # high degrees (D > 32): the readout and softmax loops make more than one lane pass over the slots, the fused row store shrinks
    # (hidden 32, D >= 72), and the readout pair lists of a hub outgrow 1024 entries (hubs_*)
    'wheel_32': wheel(32),
    'wheel_33': wheel(33),
    'wheel_72': wheel(72),
    'hubs_8x120': hubs(8, 120),
    'hubs_8x121': hubs(8, 121),
}

# The high-degree cases, what they are built to reach, and the numbers that put them there:
#   (N, E, F, D, most readout pairs of one last node (the sum of the degrees of its neighbours))
#   wheel_32    D = 32: the largest degree that starts an unfused model on the cone pipeline (3)
#   wheel_33    D = 33: one past it (the whole-support pipeline, 2), and a second lane pass in every per-slot loop
#   wheel_72    D = 72: hidden 32 shrinks the fused row store below 192 rows
#   hubs_8x120  D = 127: a hub's pair list (1849) is beyond the 1024 entries the readout kernels stage; a rim node's (1016) is not
#   hubs_8x121  D = 128: the largest degree the library supports
HIGH_DEGREE = {
    'wheel_32': (33, 64, 32, 32, 96),
    'wheel_33': (34, 66, 33, 33, 99),
    'wheel_72': (73, 144, 72, 72, 216),
    'hubs_8x120': (128, 988, 3416, 127, 1849),
    'hubs_8x121': (129, 996, 3444, 128, 1864),
}
READOUT_PAIRS_STAGED = 1024           # pair lists up to this length are staged in shared memory by the readout kernels


def readout_pairs(B1):
    """(neighbour, incident edge) pairs of the readout of a trajectory ending at each node: the sum of its neighbours' degrees."""
    A = np.abs(B1) @ np.abs(B1).T
    deg = np.abs(B1).sum(axis=1)
    np.fill_diagonal(A, 0)
    return (A > 0).astype(np.int64) @ deg.astype(np.int64)


@pytest.mark.parametrize('name', sorted(HIGH_DEGREE))
def test_high_degree_cases_are_what_they_claim(name):
    n, edges, faces = CASES[name]
    N, E, F, D, pairs = HIGH_DEGREE[name]
    assert (n, len(edges), len(faces)) == (N, E, F)
    edges, faces = np.asarray(edges, np.int64), np.asarray(faces, np.int64)
    assert np.all(edges[:, 0] < edges[:, 1]) and np.all(np.diff(faces, axis=1) > 0)
    assert len({tuple(e) for e in edges}) == E and len({tuple(f) for f in faces}) == F
    B1, B2 = so.incidence_matrices(n, edges, faces)
    assert np.abs(B1 @ B2).max() == 0
    nb, n_nbrs, _ = so.neighbourhood_tables(B1, np.arange(n))
    deg = np.abs(B1).sum(axis=1).astype(np.int64)
    assert nb.shape[1] == D == deg.max() and np.array_equal(n_nbrs, deg)
    # pair counts through the neighbour table: a trajectory ending at v reads deg(u) edges for every neighbour u of v
    by_table = np.array([deg[row[row >= 0]].sum() for row in nb])
    assert np.array_equal(by_table, readout_pairs(B1)) and by_table.max() == pairs
    if name.startswith('hubs'):
        # hubs end with more pairs than the readout kernels stage, rim nodes with fewer: both paths in one launch
        assert by_table[:8].min() > READOUT_PAIRS_STAGED >= by_table[8:].max()
    assert D <= 128                                                                  # the library's maximum degree


@pytest.mark.parametrize('model', ['scone', 'ebli'])
@pytest.mark.parametrize('name', sorted(CASES))
def test_shift_operators_and_neighbour_table_bit_exact(name, model):
    import scone_gcn_b200 as sg
    n, edges, faces = CASES[name]
    edges, faces = np.asarray(edges, np.int64).reshape(-1, 2), np.asarray(faces, np.int64).reshape(-1, 3)
    B1, B2 = so.incidence_matrices(n, edges, faces)
    if len(faces):
        assert np.abs(B1 @ B2).max() == 0                                              # boundary of a boundary
    cx = sg.SimplicialComplex.from_simplices(n, edges, faces, model, index_only=True)
    assert (cx.N, cx.E, cx.F) == (n, len(edges), len(faces))
    ref = so.shift_matrices(B1, B2, model)
    for k in range(2):
        got = cx.shift_dense(k)
        assert np.array_equal(got, np.asarray(ref[k])), (name, model, k)
        rowptr, col, _ = cx.shift_csr(k)
        for e in range(cx.E):                                                          # columns ascending: the fixed summation order
            c = col[rowptr[e]:rowptr[e + 1]]
            assert np.all(np.diff(c) > 0)
    # neighbour table: sorted neighbours, padded with -1 to the maximum degree; isolated nodes are all -1
    last_nodes = np.arange(n)
    nb, n_nbrs, _ = so.neighbourhood_tables(B1, last_nodes)
    assert cx.D == nb.shape[1] == int(np.abs(B1).sum(axis=1).max())
    assert np.array_equal(cx.nbrhoods, nb)
    assert np.array_equal((cx.nbrhoods >= 0).sum(axis=1), n_nbrs)
    # the two routes into the library agree (dense B1 / B2 as the reference stores them vs simplex lists)
    cx2 = sg.SimplicialComplex.from_dense(B1, B2, model, index_only=True)
    for k in range(2):
        assert np.array_equal(cx2.shift_dense(k), cx.shift_dense(k))
    assert sorted(np.asarray(cx.edge_rank).tolist()) == list(range(cx.E))              # internal order: a permutation

"""Ocean-drifter dataset (config 2): converter mirror vs the fixture built with the reference's own functions."""
import struct

import numpy as np
import pytest

from golden_util import Dataset, load
from scone_gcn_b200 import buoy_data

_UNDEF = 0xffffffffffffffff


def _raw(fx):
    traj = [fx['raw_traj_nodes'][fx['raw_traj_ptr'][i]:fx['raw_traj_ptr'][i + 1]].tolist() for i in range(int(fx['n_raw_traj']))]
    return fx['raw_edge_list'], fx['raw_face_list'], traj


def _write_jld2(path, datasets, contiguous=()):
    """A JLD2 file with the structure of dataBuoys.jld2 as SURVEY.md 8(f) and scone_gcn_b200/jld2.py record it: 512-byte text header,
    HDF5 superblock v2 with base address 512, v2 object headers, the root group's datasets as link messages, Int64 datasets in
    compact layout.  datasets: name -> int64 array, or list of 1-D int64 arrays (an array of object references to one compact
    dataset each, how JLD2 stores a Vector{Vector{Int64}}; the reference array is written contiguous).  Names in `contiguous` get a contiguous
    Int64 dataset instead, so that both layouts the reader supports are read.  Checksums are left zero: the reader does not check
    them."""
    body = bytearray(48)                                              # the superblock, filled in last; addresses are relative to it

    def ohdr(messages):
        msgs = b''.join(struct.pack('<BHB', t, len(d), 0) + d for t, d in messages)
        addr = len(body)
        body.extend(b'OHDR' + bytes([2, 2]) + struct.pack('<I', len(msgs)) + msgs + bytes(4))    # flags 2: 4-byte size of chunk 0
        return addr

    def dataset(arr, dtype_msg, compact):
        arr = np.ascontiguousarray(arr)
        raw = arr.astype('<u8' if dtype_msg[0] & 0x0f == 7 else '<i8').tobytes()
        if compact:
            layout = struct.pack('<BBH', 3, 0, len(raw)) + raw
        else:
            layout = struct.pack('<BBQQ', 3, 1, len(body), len(raw))
            body.extend(raw)
        space = struct.pack('<BBBB', 2, arr.ndim, 0, 1) + struct.pack('<%dQ' % arr.ndim, *arr.shape)
        return ohdr([(1, space), (3, dtype_msg), (8, layout)])

    i64 = bytes([0x10, 0x08, 0, 0]) + struct.pack('<IHH', 8, 0, 64)   # fixed-point, little-endian, signed, 64 bits
    ref = bytes([0x17, 0, 0, 0]) + struct.pack('<I', 8)              # object reference
    links = []
    for name, val in datasets.items():
        if isinstance(val, list):
            addr = dataset(np.array([dataset(np.asarray(v, np.int64), i64, True) for v in val], np.uint64), ref, False)
        else:
            addr = dataset(np.asarray(val, np.int64), i64, name not in contiguous)
        links.append((6, bytes([1, 0, len(name)]) + name.encode() + struct.pack('<Q', addr)))
    root = ohdr([(2, bytes([0, 0]) + struct.pack('<QQ', _UNDEF, _UNDEF)), (10, bytes([0, 0]))] + links)
    body[:48] = b'\x89HDF\r\n\x1a\n' + bytes([2, 8, 8, 0]) + struct.pack('<QQQQ', 512, _UNDEF, len(body), root) + bytes(4)
    with open(path, 'wb') as f:
        f.write(b'HDF5-based Julia Data Format, version 0.1.0'.ljust(512, b'\x00') + bytes(body))


def test_converter_reproduces_reference_fixture():
    fx = load('dataset_drifters.npz')
    ds = Dataset('dataset_drifters.npz')
    d = buoy_data.build_drifter_dataset(*_raw(fx))
    assert (ds.N, ds.E, ds.F, ds.D) == (133, 320, 186, 6) and len(d['paths']) == 200 and d['train_mask'].sum() == 160
    assert np.array_equal(d['B1'], ds.B1) and np.array_equal(d['B2'], ds.B2)
    assert np.array_equal(d['fwd'][0], ds.flows) and np.array_equal(d['fwd'][1], ds.targets)
    assert np.array_equal(d['fwd'][2], ds.last_nodes) and np.array_equal(d['fwd'][3], ds.target_nodes)
    assert np.array_equal(d['train_mask'], ds.train_mask)
    paths = [fx['path_nodes'][fx['path_ptr'][i]:fx['path_ptr'][i + 1]].tolist() for i in range(200)]
    assert paths == [list(map(int, p)) for p in d['paths']]


def test_jld2_reader_on_the_reference_file(tmp_path):
    """dataBuoys.jld2 is not part of the repository: its three datasets, 1-based as Julia stores them, come from the fixture (which
    holds what the reader took from the original file) and are written back with the original's structure (_write_jld2); elist is
    stored contiguous rather than compact so that the reader's other layout branch is read too."""
    fx = load('dataset_drifters.npz')
    r_el, r_fl, r_traj = _raw(fx)
    jld2 = str(tmp_path / 'dataBuoys.jld2')
    _write_jld2(jld2, {'elist': r_el + 1, 'tlist': r_fl + 1, 'TrajectoriesNodes': [np.asarray(t) + 1 for t in r_traj]},
                contiguous=('elist',))
    el, fl, traj = buoy_data.read_drifter_file(jld2)
    assert np.array_equal(el, r_el) and np.array_equal(fl, r_fl) and traj == r_traj
    d = buoy_data.convert_drifters(jld2, 'buoy', str(tmp_path))
    from scone_gcn_b200 import synthetic_data_gen as sdg
    X, (B1, B2), y, tm, sm, G, ln, tn = sdg.load_dataset(str(tmp_path / 'trajectory_data_1hop_buoy'))
    assert X.shape == (200, 320, 1) and y.shape == (200, 6, 1) and tm.sum() == 160
    assert len(np.load(str(tmp_path / 'trajectory_data_1hop_buoy' / 'prefixes.npy'), allow_pickle=True)) == 200


@pytest.mark.gpu
def test_drifter_training_matches_oracle():
    """cfg2: SCoNe on the drifter complex, 5 epochs (20 Adam steps) from 30 x the reference init (0.3-scale weights: the six
    logits are then well separated, so next-node accuracy is DECIDED): same losses, identical argmax on every trajectory whose
    oracle top-2 margin is above fp32 noise (>= 98 % of them; the rest are exact structural ties, logits equal to ~1e-7, where
    the reference's own argmax is rounding noise), accuracies equal up to those rows."""
    import scone_gcn_b200 as sg
    from oracle import scone_oracle as so
    from scone_gcn_b200.scone_trajectory_model import Scone_GCN
    from scone_gcn_b200 import trajectory_experiments as te
    import torch
    ds = Dataset('dataset_drifters.npz')
    epochs, bs, lr, wd, scale = 5, 40, 1e-3, 5e-5, 30.0
    orc = so.DenseOracle('scone', so.shift_matrices(ds.B1, ds.B2, 'scone'), ds.B1, ds.last_nodes, ds.flows, ds.targets)
    rng = np.random.RandomState(1030)
    W0 = [scale * w for w in so.generate_weights(rng, 1, [(3, 16)] * 3, 1, 'scone')]
    Wo, res_o = so.train(orc, rng, W0, ds.train_mask, ds.test_mask, epochs, bs, lr, wd)
    np.random.seed(1030)
    cx = sg.SimplicialComplex.from_dense(ds.B1, ds.B2, 'scone')
    inputs = [te.Bconds(cx), ds.last_nodes, ds.flows]
    net = Scone_GCN(epochs, lr, bs, wd, verbose=False)
    net.setup(te.scone_func, [(3, 16)] * 3, te.shift_handles(cx), inputs, ds.targets, None, ds.train_mask)
    net.weights = [scale * w for w in net.weights]
    for a, b in zip(net.weights, W0):
        assert np.array_equal(a, b)
    n_nbrs = np.array([len(so.adjacency_from_B1(ds.B1)[n]) for n in ds.last_nodes])
    res = net.train(inputs, ds.targets, ds.train_mask, ds.test_mask, n_nbrs)
    assert res[0] == pytest.approx(res_o[0], rel=2e-5) and res[2] == pytest.approx(res_o[2], rel=2e-5)
    with torch.no_grad():
        lp_o = orc.forward(Wo).numpy()[:, :, 0]
    lp = net._forward(net.weights, inputs)[:, :, 0]
    assert np.abs(lp - lp_o).max() < 2e-5 * max(1.0, np.abs(lp_o).max())
    for i in range(len(lp)):
        lp[i, n_nbrs[i]:] = -100
        lp_o[i, n_nbrs[i]:] = -100
    top2 = np.sort(lp_o, axis=1)[:, -2:]
    decided = (top2[:, 1] - top2[:, 0]) > 1e-5
    assert decided.mean() >= 0.98
    assert np.array_equal(np.argmax(lp, axis=1)[decided], np.argmax(lp_o, axis=1)[decided])
    n_tr, n_te = ds.train_mask.sum(), ds.test_mask.sum()
    assert abs(res[1] - res_o[1]) <= ((~decided) & (ds.train_mask == 1)).sum() / n_tr + 1e-9
    assert abs(res[3] - res_o[3]) <= ((~decided) & (ds.test_mask == 1)).sum() / n_te + 1e-9

"""Dense backward probe: tcgen05 backward kernel (scone_set_dense_kernel(3)) against the fp32 SIMT tile kernel (0) on the same
dense random tensors — max differences of Gprev and dW (and of dW_0 against float64), run-to-run bit-exactness, timing.
Usage: python tools/probe_bwd_umma.py [n_nodes] [b]"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import scone_gcn_b200 as sg
from scone_gcn_b200 import _lib
from scone_gcn_b200 import synthetic_data_gen as sdg

n = int(sys.argv[1]) if len(sys.argv) > 1 else 20000
b = int(sys.argv[2]) if len(sys.argv) > 2 else 64
C = 32
coords, valid, faces, edges = sdg._complex_arrays(n)
cx = sg.SimplicialComplex.from_simplices(n, edges, faces, 'scone')
L = _lib.lib()
E = cx.E
dev = torch.device('cuda')
st = torch.cuda.current_stream().cuda_stream
PEAK = 6554.2
print('complex: N=%d E=%d b=%d' % (n, E, b), flush=True)
g = torch.Generator(device='cpu').manual_seed(1)
H = torch.tanh(torch.randn(E, b, C, device=dev))
G = torch.randn(E, b, C, device=dev)
W = [torch.randn(C, C, device=dev) * 0.2 for _ in range(3)]
ws = torch.empty(L.scone_layer_backward_workspace_bytes(C, C) // 4 + 16, device=dev)


def run(which, act, with_gprev=True):
    L.scone_set_dense_kernel(which)
    Gp = torch.full((E, b, C), 7.0, device=dev) if with_gprev else None
    dW = torch.zeros(3, C, C, device=dev)
    _lib.check(L.scone_layer_backward(cx.handle, act, b, C, C, _lib.dptr(G), _lib.dptr(H), _lib.dptr(W[0]), _lib.dptr(W[1]), _lib.dptr(W[2]),
                                      _lib.dptr(Gp) if with_gprev else None, _lib.dptr(dW), 0, _lib.dptr(ws), None, None, None, None, st))
    if which == 3:
        _lib.check(L.scone_umma_status(st), 'scone_umma_status')
    torch.cuda.synchronize()
    L.scone_set_dense_kernel(_lib.DEFAULT_DENSE_KERNEL)
    return Gp, dW


def timeit(fn, iters=5, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(iters + 1)]
    ev[0].record()
    for i in range(iters):
        fn()
        ev[i + 1].record()
    torch.cuda.synchronize()
    return min(ev[i].elapsed_time(ev[i + 1]) for i in range(iters))


# float64 reference of the own-row term dW_0 = Hin^T G (the operator terms need no second opinion: same accumulation)
ref0 = torch.zeros(C, C, dtype=torch.float64, device=dev)
for lo_ in range(0, E, 8192):
    ref0 += torch.einsum('ebi,ebo->io', H[lo_:lo_ + 8192].double(), G[lo_:lo_ + 8192].double())
ok = True
for act in (0, 1, 2):
    Gp0, dW0 = run(0, act)
    Gp3, dW3 = run(3, act)
    eg = float((Gp3 - Gp0).abs().max()) / max(1.0, float(Gp0.abs().max()))
    ew = float((dW3 - dW0).abs().max()) / max(1e-30, float(dW0.abs().max()))
    Gp3b, dW3b = run(3, act)
    same = bool(torch.equal(Gp3, Gp3b) and torch.equal(dW3, dW3b))
    _, dW3n = run(3, act, with_gprev=False)
    ewn = float((dW3n - dW0).abs().max()) / max(1e-30, float(dW0.abs().max()))
    e64 = [float((x[0].double() - ref0).abs().max() / ref0.abs().max()) for x in (dW0, dW3)]
    print('   dW_0 vs float64: SIMT kernel %.2e, tcgen05 kernel %.2e' % (e64[0], e64[1]))
    print('act %d: Gprev rel err %.2e, dW rel err %.2e (no-Gprev variant %.2e), run-to-run identical %s' % (act, eg, ew, ewn, same), flush=True)
    ok = ok and eg <= 2e-5 and ew <= 2e-5 and ewn <= 2e-5 and same
print('PARITY', 'OK' if ok else 'FAIL', flush=True)
Gp = torch.empty(E, b, C, device=dev)
dW = torch.zeros(3, C, C, device=dev)
for which in (0, 3):
    L.scone_set_dense_kernel(which)
    ms = timeit(lambda: _lib.check(L.scone_layer_backward(cx.handle, 0, b, C, C, _lib.dptr(G), _lib.dptr(H), _lib.dptr(W[0]), _lib.dptr(W[1]),
                                                         _lib.dptr(W[2]), _lib.dptr(Gp), _lib.dptr(dW), 0, _lib.dptr(ws), None, None, None, None, st)))
    gbs = 4.0 * E * b * 3 * C / ms / 1e6
    print('bwd kernel=%d: %8.3f ms  %7.1f GB/s algorithmic  %.3f of %.0f' % (which, ms, gbs, gbs / PEAK, PEAK), flush=True)
L.scone_set_dense_kernel(_lib.DEFAULT_DENSE_KERNEL)

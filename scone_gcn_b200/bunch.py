"""BunchModel — owner of a `scone_bunch*` (SCCONV / "bunch" model, trajectory_experiments.py:173-203)."""
import ctypes as C

import numpy as np

from . import _lib


class CsrOperator:
    """Device-resident generic float CSR operator (`scone_csr*`) built from a scipy sparse / dense matrix."""

    def __init__(self, M):
        import scipy.sparse as sp
        M = sp.csr_matrix(M)
        M.sort_indices()
        self.shape = M.shape
        self.host = M
        rowptr = np.ascontiguousarray(M.indptr, np.int32)
        col = np.ascontiguousarray(M.indices, np.int32)
        val = np.ascontiguousarray(M.data, np.float32)
        h = C.c_void_p()
        _lib.check(_lib.lib().scone_csr_create(M.shape[0], M.shape[1], _lib.ptr(rowptr), _lib.ptr(col), _lib.ptr(val), C.byref(h)),
                   'scone_csr_create')
        self.handle = h

    def toarray(self):
        return self.host.toarray()

    def __array__(self, dtype=None, copy=None):
        a = self.toarray()
        return a if dtype is None else a.astype(dtype)

    def __del__(self):
        try:
            if getattr(self, 'handle', None):
                _lib.lib().scone_csr_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


class BunchModel:
    def __init__(self, shifts, nbrhoods, hidden, micro_batch=64):
        """shifts: 7 CsrOperator in the reference order; nbrhoods [N, D] int (pad -1); hidden: widths of the hidden layers."""
        assert len(shifts) == 7
        self.shifts = list(shifts)
        self.hidden = [int(h) for h in hidden]
        self.micro_batch = int(micro_batch)
        nb = np.ascontiguousarray(nbrhoods, np.int32)
        self.N, self.D = nb.shape
        self.E, self.F = shifts[3].shape[0], shifts[6].shape[0]
        arr = (C.c_void_p * 7)(*[s.handle for s in shifts])
        harr = np.asarray(self.hidden, np.int32)
        h = C.c_void_p()
        _lib.check(_lib.lib().scone_bunch_create(arr, self.N, self.E, self.F, self.D, _lib.ptr(nb), len(self.hidden), _lib.ptr(harr),
                                                 self.micro_batch, C.byref(h)), 'scone_bunch_create')
        self.handle = h
        self.n_params = _lib.lib().scone_bunch_num_params(h)
        widths = [1] + self.hidden + [1]
        self.shapes = []
        for i in range(len(widths) - 1):
            self.shapes += [(widths[i], widths[i + 1])] * 7

    def flatten(self, weights):
        assert len(weights) == len(self.shapes), 'wrong number of weights'
        parts = []
        for w, s in zip(weights, self.shapes):
            w = np.asarray(w, dtype=np.float32)
            assert w.shape == s, 'weight shape %s, expected %s' % (w.shape, s)
            parts.append(w.ravel())
        return np.ascontiguousarray(np.concatenate(parts))

    def unflatten(self, flat):
        out, off = [], 0
        for s in self.shapes:
            n = s[0] * s[1]
            out.append(flat[off:off + n].reshape(s).copy())
            off += n
        return out

    def set_weights(self, weights, reset_adam=True):
        flat = self.flatten(weights)
        _lib.check(_lib.lib().scone_bunch_set_weights(self.handle, _lib.ptr(flat), int(reset_adam)), 'scone_bunch_set_weights')

    def get_weights(self):
        flat = np.zeros(self.n_params, np.float32)
        _lib.check(_lib.lib().scone_bunch_get_weights(self.handle, _lib.ptr(flat)), 'scone_bunch_get_weights')
        return self.unflatten(flat)

    def forward(self, traj_ptr, flow_edge, flow_val, last_nodes, stream=None):
        B = len(last_nodes)
        out = np.zeros((B, self.D), np.float32)
        a = [np.ascontiguousarray(traj_ptr, np.int32), np.ascontiguousarray(flow_edge, np.int32),
             np.ascontiguousarray(flow_val, np.float32), np.ascontiguousarray(last_nodes, np.int32)]
        _lib.check(_lib.lib().scone_bunch_forward_host(self.handle, B, *[_lib.ptr(x) for x in a], _lib.ptr(out), stream),
                   'scone_bunch_forward_host')
        return out

    def loss_grad(self, traj_ptr, flow_edge, flow_val, last_nodes, target_idx, mask, zero_first=True, stream=None, read=True):
        B = len(last_nodes)
        a = [np.ascontiguousarray(traj_ptr, np.int32), np.ascontiguousarray(flow_edge, np.int32),
             np.ascontiguousarray(flow_val, np.float32), np.ascontiguousarray(last_nodes, np.int32),
             np.ascontiguousarray(target_idx, np.int32), np.ascontiguousarray(mask, np.float32)]
        _lib.check(_lib.lib().scone_bunch_loss_grad_host(self.handle, B, *[_lib.ptr(x) for x in a], int(zero_first), stream),
                   'scone_bunch_loss_grad_host')
        return self.read_grads(stream) if read else None

    def vjp(self, traj_ptr, flow_edge, flow_val, last_nodes, cot, count_add, zero_first=True, stream=None, read=True):
        """VJP of the log-probs (SconeModel.vjp's contract); a padded slot's cotangent reaches node N - 1, the node it reads."""
        B = len(last_nodes)
        a = [np.ascontiguousarray(traj_ptr, np.int32), np.ascontiguousarray(flow_edge, np.int32),
             np.ascontiguousarray(flow_val, np.float32), np.ascontiguousarray(last_nodes, np.int32),
             np.ascontiguousarray(cot, np.float32).reshape(B, self.D)]
        _lib.check(_lib.lib().scone_bunch_vjp_host(self.handle, B, *[_lib.ptr(x) for x in a], float(count_add), int(zero_first), stream),
                   'scone_bunch_vjp_host')
        return self.read_grads(stream) if read else None

    def read_grads(self, stream=None):
        buf = np.zeros(self.n_params + 2, np.float32)
        _lib.check(_lib.lib().scone_bunch_read_grads(self.handle, _lib.ptr(buf), stream), 'scone_bunch_read_grads')
        return buf

    def adam_step(self, step, lr, weight_decay, stream=None):
        _lib.check(_lib.lib().scone_bunch_adam_step(self.handle, int(step), float(lr), float(weight_decay), stream),
                   'scone_bunch_adam_step')

    def __del__(self):
        try:
            if getattr(self, 'handle', None):
                _lib.lib().scone_bunch_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

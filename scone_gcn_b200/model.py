"""SconeModel — owner of a `scone_model*`: device weights, Adam state, activation workspace.

Replaces vmap(scone_func / ebli_func) + grad(loss) + adam (scone_trajectory_model.py:42-56,256,300-326)."""
import ctypes as C

import numpy as np

from . import _lib


class SconeModel:
    def __init__(self, cx, hidden, micro_batch=64):
        self.cx = cx
        self.hidden = [int(h) for h in hidden]
        self.micro_batch = int(micro_batch)
        L = _lib.lib()
        harr = np.asarray(self.hidden, dtype=np.int32)
        h = C.c_void_p()
        _lib.check(L.scone_model_create(cx.handle, len(self.hidden), _lib.ptr(harr), self.micro_batch, C.byref(h)),
                   'scone_model_create')
        self.handle = h
        self.n_params = L.scone_model_num_params(h)
        self.planned = 0
        self.shapes = []
        cin = 1
        for c in self.hidden:
            self.shapes += [(cin, c)] * 3
            cin = c
        self.shapes.append((cin, 1))

    @property
    def pipeline(self):
        """0 unit kernels, 1-3 row lists (3 = readout cone), 4 = trajectory-fused kernels (include/scone_b200.h)."""
        return int(_lib.lib().scone_model_get_pipeline(self.handle))

    def set_pipeline(self, which):
        _lib.check(_lib.lib().scone_model_set_pipeline(self.handle, int(which)), 'scone_model_set_pipeline')

    def fused_info(self):
        """dict of the fused pipeline's static bounds / launch shapes, or None when the model cannot use it."""
        out = np.zeros(16, np.int32)
        _lib.check(_lib.lib().scone_model_fused_info(self.handle, _lib.ptr(out)), 'scone_model_fused_info')
        if not out[0]:
            return None
        keys = ['available', 'bound_cone', 'bound_list', 'hash_slots', 'chunk', 'cap_rows', 'plan_smem_kb', 'traj_smem_kb', 'hash_slots_tier0',
                'live_rows_tier0', 'plan_smem_tier0_kb', 'two_tiers', 'table_plan_mb', 'arena_mwords', 'cone_table_kentries', 'retries_last_chunk']
        return dict(zip(keys, (int(v) for v in out)))

    def fused_header(self, t):
        """Plan header (16 ints, csrc/fused.cuh) of trajectory t of the last chunk the fused pipeline ran."""
        hdr = np.zeros(16, np.int32)
        _lib.check(_lib.lib().scone_model_fused_read(self.handle, int(t), _lib.ptr(hdr), 0, 0, None), 'scone_model_fused_read')
        return hdr

    def check_overflow(self, stream=None):
        _lib.check(_lib.lib().scone_model_check_overflow(self.handle, stream), 'scone_model_check_overflow')

    # ---- weights ------------------------------------------------------------------------------
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

    def set_weights(self, weights, reset_adam=True, stream=None):
        flat = self.flatten(weights)
        if reset_adam:
            _lib.check(_lib.lib().scone_model_set_weights(self.handle, _lib.ptr(flat)), 'scone_model_set_weights')
        else:
            # asynchronous H2D on the caller's stream (Adam state kept); `flat` is kept alive until the next call replaces it
            self._pending_weights = flat
            _lib.check(_lib.lib().scone_model_set_weights_keep_state(self.handle, _lib.ptr(flat), stream),
                       'scone_model_set_weights_keep_state')

    def get_weights(self):
        flat = np.zeros(self.n_params, np.float32)
        _lib.check(_lib.lib().scone_model_get_weights(self.handle, _lib.ptr(flat)), 'scone_model_get_weights')
        return self.unflatten(flat)

    # ---- compute ------------------------------------------------------------------------------
    def forward(self, traj_ptr, flow_edge, flow_val, last_nodes, stream=None):
        """log-probs [B, D] (numpy) from HOST sparse flows."""
        B = len(last_nodes)
        out = np.zeros((B, self.cx.D), np.float32)
        traj_ptr = np.ascontiguousarray(traj_ptr, np.int32)
        flow_edge = np.ascontiguousarray(flow_edge, np.int32)
        flow_val = np.ascontiguousarray(flow_val, np.float32)
        last_nodes = np.ascontiguousarray(last_nodes, np.int32)
        _lib.check(_lib.lib().scone_model_forward_host(self.handle, B, _lib.ptr(traj_ptr), _lib.ptr(flow_edge),
                                                       _lib.ptr(flow_val), _lib.ptr(last_nodes), _lib.ptr(out), stream),
                   'scone_model_forward_host')
        return out

    def loss_grad(self, traj_ptr, flow_edge, flow_val, last_nodes, target_idx, mask, zero_first=True, stream=None,
                  read=True):
        """Accumulate [grads | nll_sum | count] on the device from HOST inputs; optionally read it back."""
        B = len(last_nodes)
        a = [np.ascontiguousarray(traj_ptr, np.int32), np.ascontiguousarray(flow_edge, np.int32),
             np.ascontiguousarray(flow_val, np.float32), np.ascontiguousarray(last_nodes, np.int32),
             np.ascontiguousarray(target_idx, np.int32), np.ascontiguousarray(mask, np.float32)]
        _lib.check(_lib.lib().scone_model_loss_grad_host(self.handle, B, *[_lib.ptr(x) for x in a], int(zero_first), stream),
                   'scone_model_loss_grad_host')
        return self.read_grads(stream) if read else None

    def vjp(self, traj_ptr, flow_edge, flow_val, last_nodes, cot, count_add, zero_first=True, stream=None, read=True):
        """VJP of the log-probs from HOST inputs: grads += sum cot * dlogprob/dW, nll_sum += sum cot * logprob, count += count_add, in the
        loss_grad buffer [grads | nll_sum | count]; cot [B, D] = dL/dlogprob.  Optionally read it back."""
        B = len(last_nodes)
        a = [np.ascontiguousarray(traj_ptr, np.int32), np.ascontiguousarray(flow_edge, np.int32),
             np.ascontiguousarray(flow_val, np.float32), np.ascontiguousarray(last_nodes, np.int32),
             np.ascontiguousarray(cot, np.float32).reshape(B, self.cx.D)]
        _lib.check(_lib.lib().scone_model_vjp_host(self.handle, B, *[_lib.ptr(x) for x in a], float(count_add), int(zero_first), stream),
                   'scone_model_vjp_host')
        return self.read_grads(stream) if read else None

    def vjp_flows(self, traj_ptr, flow_edge, flow_val, last_nodes, cot, count_add, zero_first=True, stream=None):
        """vjp() that also differentiates with respect to the flow values: returns (buffer, dflow), the [grads | nll_sum | count]
        buffer and dflow[p] = d(sum cot * logprob) / d flow_val[p] (float32, shaped like flow_val; entries outside
        [traj_ptr[0], traj_ptr[B]) are 0)."""
        B = len(last_nodes)
        a = [np.ascontiguousarray(traj_ptr, np.int32), np.ascontiguousarray(flow_edge, np.int32),
             np.ascontiguousarray(flow_val, np.float32), np.ascontiguousarray(last_nodes, np.int32),
             np.ascontiguousarray(cot, np.float32).reshape(B, self.cx.D)]
        dflow = np.zeros(a[2].shape, np.float32)
        _lib.check(_lib.lib().scone_model_vjp_flows_host(self.handle, B, *[_lib.ptr(x) for x in a], float(count_add), int(zero_first),
                                                         _lib.ptr(dflow), stream), 'scone_model_vjp_flows_host')
        return self.read_grads(stream), dflow

    def accuracy(self, traj_ptr, flow_edge, flow_val, last_nodes, n_nbrs, target_idx, mask, stream=None):
        """(correct, counted) over the trajectories with mask != 0: forward + argmax on the device
        (scone_trajectory_model.py:59-71; slots >= n_nbrs count as -100, first maximum wins)."""
        B = len(last_nodes)
        a = [np.ascontiguousarray(traj_ptr, np.int32), np.ascontiguousarray(flow_edge, np.int32),
             np.ascontiguousarray(flow_val, np.float32), np.ascontiguousarray(last_nodes, np.int32),
             np.ascontiguousarray(n_nbrs, np.int32), np.ascontiguousarray(target_idx, np.int32),
             np.ascontiguousarray(mask, np.float32)]
        out = np.zeros(2, np.int32)
        _lib.check(_lib.lib().scone_model_accuracy_host(self.handle, B, *[_lib.ptr(x) for x in a], _lib.ptr(out), stream),
                   'scone_model_accuracy_host')
        return int(out[0]), int(out[1])

    # ---- planned sets (pipeline 4): plan a dataset once, run only the compute kernel on rows of it every step -------------------
    def plan(self, traj_ptr, flow_edge, flow_val, last_nodes, stream=None):
        """Builds and keeps the (weight-independent) plan of these trajectories; returns False when the model has no fused pipeline."""
        if self.pipeline != 4:
            return False
        B = len(last_nodes)
        a = [np.ascontiguousarray(traj_ptr, np.int32), np.ascontiguousarray(flow_edge, np.int32),
             np.ascontiguousarray(flow_val, np.float32), np.ascontiguousarray(last_nodes, np.int32)]
        _lib.check(_lib.lib().scone_model_plan_host(self.handle, B, *[_lib.ptr(x) for x in a], stream), 'scone_model_plan_host')
        self.planned = B
        return True

    def loss_grad_planned(self, rows, target_idx, mask, zero_first=True, stream=None, read=True):
        """loss_grad over rows (indices into the planned set; None = its first len(target_idx) trajectories)."""
        n = len(target_idx)
        r = None if rows is None else np.ascontiguousarray(rows, np.int32)
        t, k = np.ascontiguousarray(target_idx, np.int32), np.ascontiguousarray(mask, np.float32)
        _lib.check(_lib.lib().scone_model_loss_grad_planned_host(self.handle, n, _lib.ptr(r), _lib.ptr(t), _lib.ptr(k), int(zero_first), stream),
                   'scone_model_loss_grad_planned_host')
        return self.read_grads(stream) if read else None

    def vjp_planned(self, rows, cot, count_add, zero_first=True, stream=None, read=True):
        """vjp over rows of the planned set (None = its first len(cot) trajectories); cot [n, D] by batch position."""
        n = len(cot)
        r = None if rows is None else np.ascontiguousarray(rows, np.int32)
        c = np.ascontiguousarray(cot, np.float32).reshape(n, self.cx.D)
        _lib.check(_lib.lib().scone_model_vjp_planned_host(self.handle, n, _lib.ptr(r), _lib.ptr(c), float(count_add), int(zero_first), stream),
                   'scone_model_vjp_planned_host')
        return self.read_grads(stream) if read else None

    def forward_planned(self, rows=None, n=None, stream=None):
        """log-probs [n, D] of rows of the planned set (None = all of it)."""
        r = None if rows is None else np.ascontiguousarray(rows, np.int32)
        n = len(r) if r is not None else (self.planned if n is None else n)
        out = np.zeros((n, self.cx.D), np.float32)
        _lib.check(_lib.lib().scone_model_forward_planned_host(self.handle, n, _lib.ptr(r), _lib.ptr(out), stream),
                   'scone_model_forward_planned_host')
        return out

    def evaluate(self, traj_ptr, flow_edge, flow_val, last_nodes, n_nbrs=None, target_idx=None, mask=None, want_choice=False,
                 want_accuracy=False, want_nll=False, stream=None):
        """Forward from HOST sparse flows with the log-probs staying on the device; returns a dict with the requested device-computed
        metrics: 'choice' [B] int32 argmax predictions, 'accuracy' (correct, counted), 'nll' (nll_sum, mask_sum)."""
        B = len(last_nodes)
        i32 = lambda a: None if a is None else np.ascontiguousarray(a, np.int32)
        a = [i32(traj_ptr), i32(flow_edge), np.ascontiguousarray(flow_val, np.float32), i32(last_nodes), i32(n_nbrs), i32(target_idx),
             None if mask is None else np.ascontiguousarray(mask, np.float32)]
        choice = np.zeros(B, np.int32) if want_choice else None
        acc = np.zeros(2, np.int32) if want_accuracy else None
        nll = np.zeros(2, np.float32) if want_nll else None
        _lib.check(_lib.lib().scone_model_eval_host(self.handle, B, *[_lib.ptr(x) for x in a], _lib.ptr(choice), _lib.ptr(acc), _lib.ptr(nll),
                                                    stream), 'scone_model_eval_host')
        out = {}
        if want_choice:
            out['choice'] = choice
        if want_accuracy:
            out['accuracy'] = (int(acc[0]), int(acc[1]))
        if want_nll:
            out['nll'] = (float(nll[0]), float(nll[1]))
        return out

    def two_target_counts(self, true_idx, rand_idx, stream=None):
        """(rows with true > random, rows with true == random) over the masked rows of the last evaluate() call."""
        B = len(true_idx)
        t, r = np.ascontiguousarray(true_idx, np.int32), np.ascontiguousarray(rand_idx, np.int32)
        out = np.zeros(2, np.int32)
        _lib.check(_lib.lib().scone_model_two_target_host(self.handle, B, _lib.ptr(t), _lib.ptr(r), _lib.ptr(out), stream),
                   'scone_model_two_target_host')
        return int(out[0]), int(out[1])

    def read_grads(self, stream=None):
        buf = np.zeros(self.n_params + 2, np.float32)
        _lib.check(_lib.lib().scone_model_read_grads(self.handle, _lib.ptr(buf), stream), 'scone_model_read_grads')
        return buf

    def read_grads_async(self, pinned, stream=None):
        """Enqueue the device -> host copy of [grads | nll_sum | count] into `pinned` (a pinned float32 torch tensor or NumPy view of
        one, n_params + 2 elements) without synchronising; the caller waits on its own event before reading it."""
        ptr = pinned.data_ptr() if hasattr(pinned, 'data_ptr') else pinned.ctypes.data
        _lib.check(_lib.lib().scone_model_read_grads_async(self.handle, ptr, stream), 'scone_model_read_grads_async')

    def adam_step(self, step, lr, weight_decay, stream=None):
        _lib.check(_lib.lib().scone_model_adam_step(self.handle, int(step), float(lr), float(weight_decay), stream),
                   'scone_model_adam_step')

    def grads_tensor(self):
        """torch view of the flat device buffer [grads | nll_sum | count] (for the NCCL all-reduce)."""
        return _wrap_device_f32(_lib.lib().scone_model_grads_dev(self.handle), self.n_params + 2)

    def weights_tensor(self):
        return _wrap_device_f32(_lib.lib().scone_model_weights_dev(self.handle), self.n_params)

    def __del__(self):
        try:
            if getattr(self, 'handle', None):
                _lib.lib().scone_model_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


class _CudaArray:
    """Minimal __cuda_array_interface__ carrier so torch can alias library-owned device memory."""

    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {'shape': (int(n),), 'typestr': '<f4', 'data': (int(ptr), False), 'version': 2}


def _wrap_device_f32(ptr, n):
    import torch
    return torch.as_tensor(_CudaArray(ptr, n), device='cuda')

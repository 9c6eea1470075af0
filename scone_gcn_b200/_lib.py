"""ctypes binding of libscone_b200.so (C ABI: include/scone_b200.h)."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


class LibraryMissing(RuntimeError):
    pass


class SconeError(RuntimeError):
    pass


def library_path():
    return os.path.join(_HERE, 'libscone_b200.so')


_i32, _i64, _f32, _vp = C.c_int32, C.c_int64, C.c_float, C.c_void_p
DEFAULT_DENSE_KERNEL = 3          # scone_set_dense_kernel: tcgen05 / TMEM where the shape allows it, slab kernels elsewhere

# name -> (restype, argtypes); every symbol include/scone_b200.h declares
SIGNATURES = {
    'scone_version': (C.c_int, []),
    'scone_last_error': (C.c_char_p, []),
    'scone_launch_count': (_i64, []),
    'scone_profile_enable': (C.c_int, [_i32]),
    'scone_profile_reset': (C.c_int, []),
    'scone_profile_read': (C.c_int, [_i32, C.POINTER(_i64), C.POINTER(C.c_double)]),
    'scone_profile_read_rows': (C.c_int, [_i32, C.POINTER(_i64)]),
    'scone_complex_create': (C.c_int, [_i32, _i32, _i32, _vp, _vp, _vp, _vp, _i32, C.POINTER(_vp)]),
    'scone_complex_create_index_only': (C.c_int, [_i32, _i32, _i32, _vp, _vp, _vp, _vp, _i32, C.POINTER(_vp)]),
    'scone_complex_destroy': (C.c_int, [_vp]),
    'scone_complex_dims': (C.c_int, [_vp] + [C.POINTER(_i32)] * 4 + [C.POINTER(_i64)] * 2),
    'scone_complex_get_shift_csr': (C.c_int, [_vp, _i32, _vp, _vp, _vp]),
    'scone_complex_get_nbrhoods': (C.c_int, [_vp, _vp]),
    'scone_complex_get_edge_rank': (C.c_int, [_vp, _vp]),
    'scone_flows_to_dense': (C.c_int, [_vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp]),
    'scone_occ_scratch_bytes': (_i64, [_vp, _i32]),
    'scone_layer_forward': (C.c_int, [_vp, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'scone_layer_backward_workspace_bytes': (_i64, [_i32, _i32]),
    'scone_layer_backward': (C.c_int, [_vp, _i32, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp]),
    'scone_readout_workspace': (_i64, [_i32, _i32]),
    'scone_readout': (C.c_int, [_vp, _i32, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _f32, _vp, _vp, _vp, _vp, _i32, _vp, _vp, _vp, _vp]),
    'scone_set_dense_kernel': (C.c_int, [_i32]),
    'scone_get_dense_kernel': (C.c_int, []),
    'scone_umma_status': (C.c_int, [_vp]),
    'scone_csr_create': (C.c_int, [_i32, _i32, _vp, _vp, _vp, C.POINTER(_vp)]),
    'scone_csr_destroy': (C.c_int, [_vp]),
    'scone_bunch_create': (C.c_int, [_vp, _i32, _i32, _i32, _i32, _vp, _i32, _vp, _i32, C.POINTER(_vp)]),
    'scone_bunch_destroy': (C.c_int, [_vp]),
    'scone_bunch_num_params': (_i64, [_vp]),
    'scone_bunch_grads_dev': (_vp, [_vp]),
    'scone_bunch_set_weights': (C.c_int, [_vp, _vp, _i32]),
    'scone_bunch_get_weights': (C.c_int, [_vp, _vp]),
    'scone_bunch_forward_host': (C.c_int, [_vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp]),
    'scone_bunch_loss_grad_host': (C.c_int, [_vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _vp]),
    'scone_bunch_vjp_host': (C.c_int, [_vp, _i32, _vp, _vp, _vp, _vp, _vp, _f32, _i32, _vp]),
    'scone_bunch_read_grads': (C.c_int, [_vp, _vp, _vp]),
    'scone_bunch_adam_step': (C.c_int, [_vp, _i32, _f32, _f32, _vp]),
    'scone_model_create': (C.c_int, [_vp, _i32, _vp, _i32, C.POINTER(_vp)]),
    'scone_model_destroy': (C.c_int, [_vp]),
    'scone_model_num_params': (_i64, [_vp]),
    'scone_model_set_pipeline': (C.c_int, [_vp, _i32]),
    'scone_model_get_pipeline': (C.c_int, [_vp]),
    'scone_model_set_weights': (C.c_int, [_vp, _vp]),
    'scone_model_get_weights': (C.c_int, [_vp, _vp]),
    'scone_model_weights_dev': (_vp, [_vp]),
    'scone_model_grads_dev': (_vp, [_vp]),
    'scone_model_forward_host': (C.c_int, [_vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp]),
    'scone_model_forward_dev': (C.c_int, [_vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp]),
    'scone_model_loss_grad_dev': (C.c_int, [_vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _vp]),
    'scone_model_loss_grad_host': (C.c_int, [_vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _vp]),
    'scone_model_vjp_dev': (C.c_int, [_vp, _i32, _vp, _vp, _vp, _vp, _vp, _f32, _i32, _vp]),
    'scone_model_vjp_host': (C.c_int, [_vp, _i32, _vp, _vp, _vp, _vp, _vp, _f32, _i32, _vp]),
    'scone_model_vjp_flows_dev': (C.c_int, [_vp, _i32, _vp, _vp, _vp, _vp, _vp, _f32, _i32, _vp, _vp]),
    'scone_model_vjp_flows_host': (C.c_int, [_vp, _i32, _vp, _vp, _vp, _vp, _vp, _f32, _i32, _vp, _vp]),
    'scone_model_vjp_planned_dev': (C.c_int, [_vp, _i32, _vp, _vp, _f32, _i32, _vp]),
    'scone_model_vjp_planned_host': (C.c_int, [_vp, _i32, _vp, _vp, _f32, _i32, _vp]),
    'scone_accuracy_dev': (C.c_int, [_i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp]),
    'scone_model_accuracy_host': (C.c_int, [_vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'scone_model_read_grads': (C.c_int, [_vp, _vp, _vp]),
    'scone_model_read_grads_async': (C.c_int, [_vp, _vp, _vp]),
    'scone_model_eval_host': (C.c_int, [_vp, _i32] + [_vp] * 10 + [_vp]),
    'scone_model_two_target_host': (C.c_int, [_vp, _i32, _vp, _vp, _vp, _vp]),
    'scone_model_adam_step': (C.c_int, [_vp, _i32, _f32, _f32, _vp]),
    'scone_dp_create': (C.c_int, [_i32, _i32, _i64, C.POINTER(_vp)]),
    'scone_dp_handle_bytes': (_i32, []),
    'scone_dp_get_handle': (C.c_int, [_vp, _vp]),
    'scone_dp_open': (C.c_int, [_vp, _vp]),
    'scone_model_dp_adam_step': (C.c_int, [_vp, _vp, _i32, _f32, _f32, _vp]),
    'scone_dp_status': (C.c_int, [_vp, _vp]),
    'scone_dp_destroy': (None, [_vp]),
    'scone_model_check_overflow': (C.c_int, [_vp, _vp]),
    'scone_model_plan_host': (C.c_int, [_vp, _i32, _vp, _vp, _vp, _vp, _vp]),
    'scone_model_plan_dev': (C.c_int, [_vp, _i32, _vp, _vp, _vp, _vp, _vp]),
    'scone_model_loss_grad_planned_host': (C.c_int, [_vp, _i32, _vp, _vp, _vp, _i32, _vp]),
    'scone_model_loss_grad_planned_dev': (C.c_int, [_vp, _i32, _vp, _vp, _vp, _i32, _vp]),
    'scone_model_forward_planned_host': (C.c_int, [_vp, _i32, _vp, _vp, _vp]),
    'scone_model_set_weights_keep_state': (C.c_int, [_vp, _vp, _vp]),
    'scone_model_fused_info': (C.c_int, [_vp, _vp]),
    'scone_model_fused_read': (C.c_int, [_vp, _i32, _vp, C.c_uint32, _i32, _vp]),
    'scone_model_read_rows_done': (C.c_int, [_vp, _vp]),
}


def lib():
    """Load the CUDA library, or fail loudly (there is no CPU path)."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = library_path()
    if not os.path.exists(path):
        raise LibraryMissing(
            '%s not found: build it with `python __graft_entry__.py build` (or `make`). '
            'scone_gcn_b200 has no CPU fallback.' % path)
    L = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        f = getattr(L, name)
        f.restype, f.argtypes = res, args
    _LIB = L
    return L


def check(rc, what=''):
    if rc != 0:
        msg = lib().scone_last_error().decode('utf-8', 'replace')
        raise SconeError('%s failed (code %d): %s' % (what or 'scone call', rc, msg))


def ptr(a):
    """Host pointer of a C-contiguous numpy array (or None)."""
    if a is None:
        return None
    assert a.flags['C_CONTIGUOUS']
    return a.ctypes.data_as(C.c_void_p)


def dptr(t):
    """Device pointer of a torch CUDA tensor, a raw int address, or None."""
    if t is None:
        return None
    if isinstance(t, int):
        return C.c_void_p(t)
    assert t.is_cuda and t.is_contiguous()
    return C.c_void_p(t.data_ptr())

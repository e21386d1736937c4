"""ctypes binding of libmadstereo.so (C ABI declared in include/madstereo.h).

There is deliberately NO fallback: if the shared library is missing or a call fails the error is raised.
"""
import ctypes
import os
from ctypes import c_char_p, c_float, c_int, c_size_t, c_void_p, POINTER

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(os.path.dirname(_HERE), 'libmadstereo.so')
_lib = None


class MadStereoError(RuntimeError):
    pass


P = c_void_p
I = c_int
F = c_float
Z = c_size_t

_SIGS = {
    'ms_version': (I, []),
    'ms_last_error': (c_char_p, []),
    'ms_corr_fwd': (I, [P, I, P, I, P, I, P, I, I, I, I, I, I, I, I, I, P]),
    'ms_debug_mma_probe': (I, [I, I, I, I, I, I, I, I, P, P]),
    'ms_corr_fwd_wide': (I, [P, I, P, I, P, I, I, I, I, I, I, F, P]),
    'ms_corr_bwd': (I, [P, I, P, I, P, I, P, I, P, I, P, I, P, I, I, I, I, I, I, I, I, P]),
    'ms_conv2d_fwd': (I, [P, I, I, I, I, I, P, P, P, I, I, I, I, I, I, F, P]),
    'ms_conv2d_dgrad': (I, [P, I, I, I, I, I, P, P, I, I, I, I, I, I, I, I, P, P]),
    'ms_conv2d_fwd_bf': (I, [P, I, I, I, I, I, P, P, P, I, I, I, I, I, I, F, F, P, Z, P]),
    'ms_conv2d_dgrad_bf': (I, [P, I, I, I, I, I, P, P, I, I, I, I, I, I, I, I, P, Z, P]),
    'ms_conv2d_bf_scratch': (Z, [I, I, I, I, I, I, I]),
    'ms_conv2d_wgrad_bf': (I, [P, I, I, I, I, I, P, I, I, I, I, P, P, I, I, I, I, P, Z, P]),
    'ms_conv2d_wgrad_bf_scratch': (Z, [I, I, I, I, I, I, I, I, I]),
    'ms_bf_split': (I, [P, I, I, I, I, I, P, P, I, I, F, P]),
    'ms_bf_weight_halfs': (Z, [I, I, I]),
    'ms_bf_prep_weights': (I, [P, I, I, I, I, I, P, P, P]),
    'ms_conv2d_fwd_bf_planes': (I, [P, P, I, I, F, I, I, I, I, P, P, P, I, I, P, P, I, I, I, I, I, F, P, P, P]),
    'ms_conv2d_bf_part_floats': (Z, []),
    'ms_conv2d_bf_ticket_words': (Z, []),
    'ms_conv2d_wgrad_bf_planes': (I, [P, P, I, I, I, I, I, P, P, I, I, I, I, P, P, I, I, I, I, P, Z, P]),
    'ms_conv2d_wgrad_bf_workspace': (Z, [I, I, I, I]),
    'ms_conv2d_wgrad_tc': (I, [P, I, I, I, I, I, P, I, I, P, P, I, I, I, P, Z, P]),
    'ms_conv2d_wgrad_tc_workspace': (Z, [I, I, I, I, I, I, I]),
    'ms_conv2d_wgrad_workspace': (Z, [I, I, I, I, Z]),
    'ms_conv2d_wgrad': (I, [P, I, I, I, I, I, P, I, I, I, I, P, P, I, I, I, I, P, Z, P]),
    'ms_conv2d_transpose_fwd': (I, [P, I, I, I, I, I, P, P, P, I, I, I, I, I, F, P, P]),
    'ms_conv2d_stem_fwd': (I, [P, I, I, I, P, P, P, I, F, P]),
    'ms_conv2d_stem_wgrad_workspace': (Z, [I, I, I]),
    'ms_conv2d_stem_wgrad': (I, [P, I, I, I, P, I, P, P, P, Z, P]),
    'ms_conv2d_transpose_fwd_bf': (I, [P, I, I, I, I, I, P, P, P, I, I, I, I, I, F, F, P, Z, P]),
    'ms_conv2d_transpose_dgrad_bf': (I, [P, I, I, I, I, I, P, P, I, I, I, I, I, P, Z, P]),
    'ms_conv2d_transpose_bf_scratch': (Z, [I, I, I, I, I, I, I, I]),
    'ms_conv2d_transpose_wgrad_bf': (I, [P, I, I, I, I, I, P, I, I, P, P, I, I, I, P, Z, P]),
    'ms_conv2d_transpose_wgrad_bf_scratch': (Z, [I, I, I, I, I, I, I, I]),
    'ms_resize_bilinear': (I, [P, I, I, I, I, P, I, I, I, I, I, F, I, F, I, P]),
    'ms_resize_bilinear_bwd': (I, [P, I, P, I, I, I, I, P, I, I, I, I, I, F, I, F, I, I, P, P]),
    'ms_reproj_loss_workspace': (Z, [I, I, I]),
    'ms_reproj_loss': (I, [P, P, P, I, I, I, P, P, P, F, P]),
    'ms_momentum_update': (I, [P, P, P, Z, F, F, F, P]),
    'ms_pad_reflect': (I, [P, I, I, I, I, P, I, I, I, F, F, P]),
    'ms_engine_create': (P, [c_char_p, I, I, I, I, I, I]),
    'ms_engine_destroy': (I, [P]),
    'ms_engine_num_layers': (I, [P]),
    'ms_engine_layer_info': (I, [P, I, c_char_p, I, c_char_p, I, c_char_p, I, POINTER(I), POINTER(F)]),
    'ms_engine_set_groups': (I, [P, POINTER(I), I, I]),
    'ms_engine_sizes': (I, [P, POINTER(Z), POINTER(Z)]),
    'ms_engine_param_offsets': (I, [P, I, POINTER(Z), POINTER(Z)]),
    'ms_engine_group_range': (I, [P, I, POINTER(Z), POINTER(Z)]),
    'ms_engine_bind': (I, [P, P, P, P, P, Z, P]),
    'ms_engine_set_input': (I, [P, P, P, P]),
    'ms_engine_set_input_u8': (I, [P, P, P, P]),
    'ms_engine_set_gt': (I, [P, P, P]),
    'ms_engine_set_proxy': (I, [P, P, P]),
    'ms_engine_set_loss': (I, [P, I, F, F]),
    'ms_engine_dp_create': (I, [P, I, I, P]),
    'ms_engine_dp_connect': (I, [P, P]),
    'ms_engine_dp_error': (I, [P, P]),
    'ms_engine_forward': (I, [P, I, P]),
    'ms_engine_loss': (I, [P, I, I, I, F, P]),
    'ms_engine_backward': (I, [P, I, I, P]),
    'ms_engine_update': (I, [P, I, F, F, F, P]),
    'ms_engine_run': (I, [P, I, I, I, I, F, F, F, P]),
    'ms_engine_weights_changed': (I, [P]),
    'ms_engine_read_scalars': (I, [P, POINTER(F), P]),
    'ms_engine_metrics': (I, [P, P]),
    'ms_engine_profile': (I, [P, I]),
    'ms_engine_profile_read': (I, [P, POINTER(ctypes.c_double), POINTER(ctypes.c_double), POINTER(ctypes.c_double), POINTER(ctypes.c_longlong)]),
    'ms_engine_profile_layers': (I, [P, P, P]),
    'ms_engine_profile_event_overhead_ms': (F, [P]),
    'ms_launch_count': (ctypes.c_longlong, []),
    'ms_debug_bf_prof': (I, [P, I]),
    'ms_engine_num_tensors': (I, [P]),
    'ms_engine_tensor_name': (I, [P, I, c_char_p, I]),
    'ms_engine_tensor': (I, [P, c_char_p, POINTER(P), POINTER(I)]),
}

EXPORTS = sorted(_SIGS)


def lib():
    """Load (once) and return the ctypes handle; raises MadStereoError when the library is absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise MadStereoError(
                'libmadstereo.so not found at %s - build it with `make -C csrc` or __graft_entry__.build(); '
                'there is no CPU / PyTorch fallback' % LIB_PATH)
        h = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(h, name)
            fn.restype = res
            fn.argtypes = args
        _lib = h
    return _lib


def check(rc, what=''):
    if rc != 0:
        msg = lib().ms_last_error()
        raise MadStereoError('%s failed (%d): %s' % (what, rc, msg.decode() if msg else '?'))

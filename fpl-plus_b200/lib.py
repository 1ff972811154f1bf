"""ctypes binding of libfplplus_b200.so (the C ABI declared in include/fplplus_b200.h).

There is deliberately no fallback: if the library is missing it is built with nvcc, and if
that is impossible the import fails loudly.
"""
import ctypes
from ctypes import c_char_p, c_double, c_float, c_int, c_int64, c_longlong, c_uint64, c_void_p

from . import build as _build

_P = c_void_p
_I = c_int
_L = c_int64
_F = c_float
_U = c_uint64

_SIGNATURES = {
    "fpl_last_error": (c_char_p, []),
    "fpl_version": (_I, []),
    "fpl_set_sm_budget": (_I, [_I]),
    "fpl_launch_count": (c_longlong, [_I]),
    "fpl_device_is_sm100": (_I, []),
    "fpl_conv3d_weight_image_bytes": (_L, [_I, _I, _I]),
    "fpl_conv3d_prep_weight": (_I, [_P, _I, _I, _I, _I, _P, _P]),
    "fpl_conv3d_prep_weight_batch": (_I, [_I, ctypes.POINTER(c_void_p), ctypes.POINTER(_I), ctypes.POINTER(_I),
                                          ctypes.POINTER(_I), ctypes.POINTER(_I), ctypes.POINTER(c_void_p), _P]),
    "fpl_conv3d_tc": (_I, [_P, _I, _I, _P, _P, _P, _I, _I, _P] + [_I] * 7 + [_P]),
    "fpl_conv3d_dfold_image_bytes": (_L, [_I, _I]),
    "fpl_conv3d_dfold_prep_weight": (_I, [_P, _I, _I, _I, _P, _P]),
    "fpl_conv3d_dfold_prep_weight_batch": (_I, [_I, ctypes.POINTER(c_void_p), ctypes.POINTER(_I), ctypes.POINTER(_I),
                                                ctypes.POINTER(_I), ctypes.POINTER(c_void_p), _P]),
    "fpl_conv3d_tc_dfold": (_I, [_P, _I, _I, _P, _P, _P, _I, _I, _P] + [_I] * 6 + [_P]),
    "fpl_patch9_c8": (_I, [_P, _P, _I, _I, _I, _I, _I, _P]),
    "fpl_conv3d_k311_prep_weight": (_I, [_P, _I, _I, _P, _P]),
    "fpl_conv3d_tc_k311": (_I, [_P, _I, _I, _P, _P, _P, _I, _I, _P] + [_I] * 7 + [_P]),
    "fpl_conv3d_wgrad_tc_k311": (_I, [_P, _I, _I, _P, _I, _I, _P] + [_I] * 6 + [_P]),
    "fpl_conv3d_direct": (_I, [_P, _I, _I, _P, _P, _P, _I, _I, _P] + [_I] * 9 + [_P]),
    "fpl_conv3d_wgrad": (_I, [_P, _I, _I, _P, _I, _I, _P] + [_I] * 7 + [_P]),
    "fpl_conv3d_wgrad_tc": (_I, [_P, _I, _I, _P, _I, _I, _P] + [_I] * 7 + [_P]),
    "fpl_conv3d_wgrad_tc_tapmajor": (_I, [_P, _I, _I, _P, _I, _I, _P] + [_I] * 7 + [_P]),
    "fpl_wgrad_tapmajor_to_dw_batch": (_I, [_I, ctypes.POINTER(c_void_p), ctypes.POINTER(c_void_p), ctypes.POINTER(_I),
                                            ctypes.POINTER(_I), ctypes.POINTER(_I), ctypes.POINTER(_I), _P]),
    "fpl_dsbn_eval_affine_batch": (_I, [_I] + [ctypes.POINTER(c_void_p)] * 7 + [ctypes.POINTER(_I), _F, _P]),
    "fpl_conv3d_tc_act": (_I, [_P, _I, _I, _P, _P, _I, _I] + [_I] * 7 + [_P, _P, _P, _F, _U, _U, _P, _P]),
    "fpl_conv3d_tc_dfold_act": (_I, [_P, _I, _I, _P, _P, _I, _I] + [_I] * 6 + [_P, _P, _P, _P]),
    "fpl_conv3d_tc_k311_act": (_I, [_P, _I, _I, _P, _P, _I, _I] + [_I] * 7 + [_P, _P, _P, _P]),
    "fpl_maxpool_c8": (_I, [_P, _I, _I, _P, _I, _I, _I] + [_I] * 5 + [_P]),
    "fpl_head_fwd": (_I, [_P, _I, _I, _P, _P, _P] + [_I] * 6 + [_P]),
    "fpl_head_dgrad": (_I, [_P, _P, _P, _I, _I, _P, _I, _I, _P] + [_I] * 6 + [_P]),
    "fpl_upsample2x_c8": (_I, [_P, _I, _I, _P, _I, _I] + [_I] * 6 + [_P]),
    "fpl_upsample2x_c8_bwd": (_I, [_P, _I, _I, _P, _I, _I] + [_I] * 6 + [_P]),
    "fpl_channel_sum_c8": (_I, [_P, _I, _I, _P] + [_I] * 5 + [_P]),
    "fpl_grad_scatter_add": (_I, [_P, _P, _P, _I, _I, _P]),
    "fpl_stem_conv_fwd": (_I, [_P, _P, _P, _P, _I, _I, _P] + [_I] * 7 + [_P]),
    "fpl_stem_conv_wgrad": (_I, [_P, _P, _I, _I, _P] + [_I] * 7 + [_P]),
    "fpl_head_conv_fwd": (_I, [_P, _I, _I, _P, _P, _P] + [_I] * 6 + [_P]),
    "fpl_head_conv_tc": (_I, [_P, _I, _I, _P, _P, _P] + [_I] * 6 + [_P]),
    "fpl_pack_ncdhw_to_c8": (_I, [_P, _I, _P, _I, _I, _I, _P] + [_I] * 4 + [_P]),
    "fpl_head_conv_bwd": (_I, [_P, _I, _I, _P, _P, _P, _I, _I, _P, _P] + [_I] * 6 + [_P]),
    "fpl_convt_k2s2_fwd": (_I, [_P, _I, _I, _P, _P, _P, _I, _I] + [_I] * 7 + [_P]),
    "fpl_convt_k2s2_bwd": (_I, [_P, _I, _I, _P, _P, _I, _I, _P, _I, _I, _P, _P] + [_I] * 7 + [_P]),
    "fpl_convt_weight_image_bytes": (_L, [_I, _I, _I]),
    "fpl_convt_prep_weight": (_I, [_P, _I, _I, _I, _I, _P, _P]),
    "fpl_convt_prep_weight_batch": (_I, [_I, ctypes.POINTER(c_void_p), ctypes.POINTER(_I), ctypes.POINTER(_I),
                                         ctypes.POINTER(_I), ctypes.POINTER(_I), ctypes.POINTER(c_void_p), _P]),
    "fpl_convt_k2s2_fwd_tc": (_I, [_P, _I, _I, _P, _P, _P, _I, _I] + [_I] * 7 + [_P]),
    "fpl_convt_k2s2_dgrad_tc": (_I, [_P, _I, _I, _P, _P, _I, _I] + [_I] * 7 + [_P]),
    "fpl_convt_k2s2_wgrad_tc": (_I, [_P, _I, _I, _P, _I, _I, _P] + [_I] * 7 + [_P]),
    "fpl_convt_k2s2_wgrad_tc_tapmajor": (_I, [_P, _I, _I, _P, _I, _I, _P] + [_I] * 7 + [_P]),
    "fpl_dsbn_finalize": (_I, [_P, _L, _P, _P, _P, _P, _P, _F, _F, _I, _P, _P, _P, _P, _I, _P]),
    "fpl_dsbn_act_fwd": (_I, [_P, _P, _P, _P, _P, _I, _I, _P, _I, _I, _P, _I, _F, _P, _U, _U, _P] + [_I] * 5 + [_P]),
    "fpl_dsbn_bn_act_fwd": (_I, [_P, _P, _L, _P, _P, _P, _P, _P, _F, _F, _I, _P, _P, _P, _P, _P,
                                 _P, _I, _I, _P, _I, _I, _P, _I, _F, _P, _U, _U, _P] + [_I] * 5 + [_P]),
    "fpl_dsbn_act_bwd_apply_fin": (_I, [_P, _P, _I, _I, _P, _I, _I, _P, _I, _P, _P, _P, _P, _P, _F, _P, _U, _U, _P, _P, _I, _P]
                                   + [_I] * 5 + [_P, _P, _P, _P, _P]),
    "fpl_dsbn_act_bwd_reduce": (_I, [_P, _P, _I, _I, _P, _I, _I, _P, _I, _P, _P, _P, _P, _P, _F, _P, _U, _U, _P, _P]
                                + [_I] * 5 + [_P]),
    "fpl_dsbn_act_bwd_apply": (_I, [_P, _P, _I, _I, _P, _I, _I, _P, _I, _P, _P, _P, _P, _P, _F, _P, _U, _U, _P, _P, _I, _P]
                               + [_I] * 5 + [_P]),
    "fpl_dsbn_bwd_finalize": (_I, [_P, _P, _P, _I, _P, _P, _P, _P, _I, _P]),
    "fpl_gather_patches": (_I, [_P, _I, _I, _I, _I, _I, _P, _P, _P, _P]),
    "fpl_gather_patches_norm_workspace_bytes": (_L, [_I] * 5),
    "fpl_gather_patches_norm": (_I, [_P, _I, _I, _I, _I, _I, ctypes.POINTER(_I), ctypes.POINTER(_F), ctypes.POINTER(_F), _P,
                                     _L, _P, _P, _P, _P]),
    "fpl_adam_multi_tensor": (_I, [_P, _I, _P, _I, _P, c_double, c_double, c_double, c_double, c_double, _P, _P]),
    "fpl_adam_chunk_elems": (_I, []),
    "fpl_dice_ce_reduce": (_I, [_P, _P, _P, _P, _I, _I, _L, _P]),
    "fpl_dice_ce_grad": (_I, [_P, _P, _P, _P, _F, _F, _F, _P, _P, _P, _I, _I, _L, _P]),
    "fpl_dice_ce_reduce_ex": (_I, [_P, _P, _P, _P, _P, _P, _P, _I, _I, _L, _I, _I, _P]),
    "fpl_dice_ce_grad_ex": (_I, [_P, _P, _P, _P, _P, _P, _P, _F, _F, _F, _F, _P, _P, _P, _I, _I, _L, _I, _I, _P]),
    "fpl_dice_ce_loss_ex": (_I, [_P, _P, _P, _P, _P, _P, _P, _F, _F, _F, _P, _P, _I, _I, _L, _I, _I, _P]),
    "fpl_argmax_label": (_I, [_P, _P, _I, _I, _L, _P]),
    "fpl_mc_uncertainty": (_I, [ctypes.POINTER(c_void_p), _I, _I, _L, _P, _P, _P]),
    "fpl_mc_uncertainty_max_passes": (_I, []),
    "fpl_agree_weight": (_I, [_P, _P, _P, _P, _P, _I, _F, _P, _I, _L, _P]),
    "fpl_window_accumulate": (_I, [_P, _P, _P] + [_I] * 13 + [_F, _P]),
    "fpl_window_normalize": (_I, [_P, _P, _F, _L, _P]),
}

#: every symbol include/fplplus_b200.h declares (tests check the .so exports them all)
EXPORTED = list(_SIGNATURES)

_lib = None


class FplError(RuntimeError):
    pass


def load():
    global _lib
    if _lib is None:
        path = _build.build()
        lib = ctypes.CDLL(path)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


#: optional per-call instrumentation: a callable(name, args) -> context token with .stop(); bench.py
#: installs one that brackets selected entry points with CUDA events on the launching stream
_call_timer = None


def set_call_timer(fn):
    global _call_timer
    _call_timer = fn


def call(name, *args):
    """Invoke a C-ABI function; a non-zero status raises FplError with the library's message."""
    lib = load()
    tok = _call_timer(name, args) if _call_timer is not None else None
    rc = getattr(lib, name)(*args)
    if tok is not None:
        tok.stop()
    if rc != 0:
        raise FplError("%s failed (%d): %s" % (name, rc, lib.fpl_last_error().decode()))


def launch_count(reset=False):
    return int(load().fpl_launch_count(1 if reset else 0))

"""ctypes binding of the C ABI declared in include/damvs.h.

There is no fallback: if the shared library has not been built, importing any
compute entry point raises.  ``python -m damvsnet_b200.build`` builds it.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_longlong, c_size_t, c_uint64, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "_C", "libdamvs_b200.so")

F32, BF16, F16 = 0, 1, 2
AGG_VARIANCE, AGG_ADAPTIVE = 0, 1
CONV_DIRECT, CONV_TCGEN05 = 0, 1


class ConvDesc(ctypes.Structure):
    """Mirror of ``damvs_conv3d_desc`` (include/damvs.h)."""
    _fields_ = [(n, c_int) for n in ("B", "Cin", "Cout", "Din", "Hin", "Win", "stride", "transposed", "relu",
                                     "in_dtype", "out_dtype", "plain_out", "impl")]


_SIGNATURES = {
    "damvs_abi_version": (c_int, []),
    "damvs_last_error": (c_char_p, []),
    "damvs_check_device": (c_int, [c_int]),
    "damvs_nchw_to_nhwc_f32": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "damvs_ncdhw_to_g8": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "damvs_g8_to_ncdhw": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "damvs_homo_warp_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int,
                                    c_void_p]),
    "damvs_warp_agg_fwd": (c_int, [c_void_p, POINTER(c_void_p), c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                   c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "damvs_nchw_to_nhwc_f16": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "damvs_nchw_to_nhwc_f16_multi": (c_int, [POINTER(c_void_p), POINTER(c_void_p), c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "damvs_warp_agg_fwd_f16": (c_int, [c_void_p, POINTER(c_void_p), c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                       c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "damvs_warp_gwc_fwd": (c_int, [c_void_p, POINTER(c_void_p), c_int, c_void_p, c_void_p, c_void_p] + [c_int] * 9 + [c_void_p]),
    "damvs_warp_gwc_train_fwd": (c_int, [c_void_p, POINTER(c_void_p), c_int, c_void_p, c_void_p, c_void_p] + [c_int] * 8
                                 + [c_void_p]),
    "damvs_warp_gwc_bwd": (c_int, [c_void_p, POINTER(c_void_p), c_int, c_void_p, c_void_p, c_void_p, c_int, c_void_p,
                                   POINTER(c_void_p)] + [c_int] * 7 + [c_void_p]),
    "damvs_conv3d_packed_weight_bytes": (c_size_t, [POINTER(ConvDesc)]),
    "damvs_conv3d_pack_weight": (c_int, [POINTER(ConvDesc), c_void_p, c_void_p, c_void_p]),
    "damvs_conv3d_fwd": (c_int, [POINTER(ConvDesc), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                 c_void_p]),
    "damvs_prob_head_supported": (c_int, [POINTER(ConvDesc)]),
    "damvs_prob_head_fwd": (c_int, [POINTER(ConvDesc)] + [c_void_p] * 8),
    "damvs_softmax_regress_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                          c_int, c_int, c_int, c_void_p]),
    "damvs_depth_regression_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "damvs_softmax_regress_bwd": (c_int, [c_void_p] * 8 + [c_int] * 5 + [c_void_p]),
    "damvs_bn_stats": (c_int, [c_void_p] + [c_int] * 6 + [c_void_p, c_void_p]),
    "damvs_bn_apply": (c_int, [c_void_p] * 5 + [c_int] * 7 + [c_void_p]),
    "damvs_bn_bwd": (c_int, [c_void_p] * 9 + [c_int] * 7 + [c_void_p]),
    "damvs_bn_finalize": (c_int, [c_void_p] * 5 + [c_double, c_float, c_float] + [c_void_p] * 4 + [c_int, c_void_p]),
    "damvs_bn_bwd_coeffs": (c_int, [c_void_p] * 4 + [c_double] + [c_void_p] * 5 + [c_int, c_void_p]),
    "damvs_plain_to_g8": (c_int, [c_void_p, c_void_p, c_int, c_longlong, c_void_p]),
    "damvs_conv3d_wgrad": (c_int, [POINTER(ConvDesc), c_void_p, c_void_p, c_void_p, c_void_p]),
    "damvs_warp_agg_bwd": (c_int, [c_void_p, POINTER(c_void_p), c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p,
                                   POINTER(c_void_p), c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "damvs_warp_score_fwd": (c_int, [c_void_p, POINTER(c_void_p), c_int, c_void_p, c_void_p, c_void_p, c_void_p] + [c_int] * 6
                             + [c_void_p]),
    "damvs_warp_weighted_fwd": (c_int, [c_void_p, POINTER(c_void_p), c_int, c_void_p, c_void_p, c_void_p, c_void_p]
                                + [c_int] * 7 + [c_void_p]),
    "damvs_uncertainty_samples_fwd": (c_int, [c_void_p, c_void_p, c_void_p] + [c_int] * 7 + [c_void_p]),
    "damvs_geo_consistency_fuse": (c_int, [c_void_p] * 4 + [POINTER(c_void_p), POINTER(c_double), c_int, c_int, c_int, c_float, c_float, c_float,
                                           c_double, c_double] + [c_void_p] * 5),
    "damvs_cross_view_terms": (c_int, [c_void_p, c_void_p, POINTER(c_void_p), c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "damvs_cross_view_select": (c_int, [c_void_p, c_void_p, c_int, c_longlong, c_void_p, c_void_p]),
    "damvs_cross_view_bwd": (c_int, [c_void_p, c_void_p, POINTER(c_void_p), c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "damvs_warp_gwt": (c_int, [c_void_p, POINTER(c_void_p), c_int, c_void_p, c_void_p, c_void_p, c_int, c_void_p] + [c_int] * 6 + [c_void_p]),
    "damvs_warp_merged_bwd": (c_int, [c_void_p, POINTER(c_void_p), c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int,
                                      c_void_p, POINTER(c_void_p), c_void_p] + [c_int] * 6 + [c_void_p]),
    "damvs_wnet_chain_fwd": (c_int, [c_void_p, c_int, c_longlong, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                     c_void_p, c_float, c_float, c_void_p, c_void_p, c_void_p, c_void_p]),
    "damvs_wnet_chain_bwd": (c_int, [c_void_p, c_void_p, c_int, c_longlong, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "damvs_launch_count": (c_uint64, []),
}

EXPORTS = tuple(_SIGNATURES)

_lib = None


def load() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"damvsnet_b200: CUDA library {LIB_PATH} is missing. Build it with `python -m damvsnet_b200.build` "
            "(needs nvcc; sm_100a only). There is no CPU or PyTorch fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.damvs_abi_version() != 1:
        raise RuntimeError("damvsnet_b200: ABI version mismatch between _lib.py and the built library")
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        msg = load().damvs_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"damvs error {rc}: {msg}")


def launch_count() -> int:
    return int(load().damvs_launch_count())

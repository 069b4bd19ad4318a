"""ctypes binding of libpcgc_b200.so (the C ABI in include/pcgc_b200.h).

This is the stub a maintainer of the reference would add next to ``transform.py`` (see
INTEGRATION.md).  There is NO CPU fallback: if the library is missing or a device call fails the
product raises ``RuntimeError``; the oracle under ``oracle/`` is test infrastructure and is never
imported from here.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PCGC_LIB") or os.path.join(_HERE, "libpcgc_b200.so")   # PCGC_LIB: dev hook (A/B builds of one kernel, tools/)

# enums of include/pcgc_b200.h
NET_VOX_ANALYSIS, NET_VOX_SYNTHESIS, NET_HYPER_ENCODER, NET_HYPER_DECODER, NET_SIMPLE_ANALYSIS, NET_SIMPLE_SYNTHESIS = range(6)
DTYPE_U8, DTYPE_F32, DTYPE_F64 = range(3)
MESH_OBJ, MESH_OFF, MESH_PLY = range(3)
ENGINE_AUTO, ENGINE_FFMA, ENGINE_UMMA = range(3)
MAX_SYMBOLS = 64
ERR_BAD_ARG, ERR_BAD_RANGE, ERR_CUDA, ERR_OOM, ERR_NOT_READY, ERR_OVERFLOW, ERR_CORRUPT = -1, -2, -3, -4, -5, -6, -7
ERR_NAMES = {0: "OK", -1: "BAD_ARG", -2: "BAD_RANGE", -3: "CUDA", -4: "OOM", -5: "NOT_READY", -6: "OVERFLOW", -7: "CORRUPT"}

_vp, _i, _i64, _f = C.c_void_p, C.c_int, C.c_int64, C.c_float

# name -> (restype, argtypes); must list EVERY symbol the header declares (tests check this)
SIGNATURES = {
    "pcgc_abi_version": (_i, []),
    "pcgc_create": (_i, [C.POINTER(_vp), _i]),
    "pcgc_destroy": (None, [_vp]),
    "pcgc_last_error": (C.c_char_p, [_vp]),
    "pcgc_set_stream": (_i, [_vp, _vp]),
    "pcgc_set_engine": (_i, [_vp, _i]),
    "pcgc_launch_count": (_i64, [_vp]),
    "pcgc_synchronize": (_i, [_vp]),
    "pcgc_profile_enable": (_i, [_vp, _i]),
    "pcgc_profile_report": (_i, [_vp, C.c_char_p, _i64]),
    "pcgc_load_conv": (_i, [_vp, _i, C.c_char_p, _vp, C.POINTER(_i64), _vp]),
    "pcgc_load_bottleneck": (_i, [_vp, _i, _i, _vp, _vp, _vp]),
    "pcgc_debug_conv3_umma": (_i, [_vp, _vp, _i, _i, _i, _vp, _vp, _i, _i, _i, _vp]),
    "pcgc_analysis": (_i, [_vp, _i, _vp, _i, _i, _vp]),
    "pcgc_synthesis": (_i, [_vp, _i, _vp, _i, _vp]),
    "pcgc_hyper_encode": (_i, [_vp, _vp, _i, _vp]),
    "pcgc_hyper_decode": (_i, [_vp, _vp, _i, _f, _vp, _vp]),
    "pcgc_factorized_quantize_likelihood": (_i, [_vp, _i, _vp, _i64, _i, _f, _vp, _vp, _vp, _vp]),
    "pcgc_factorized_cdf": (_i, [_vp, _i, _i, _i, _f, _i, _vp]),
    "pcgc_laplace_quantize_likelihood": (_i, [_vp, _vp, _vp, _vp, _i, _i64, _f, _vp, _vp, _vp, _vp]),
    "pcgc_widen_symbol_ranges": (_i, [_vp, _vp, _i]),
    "pcgc_laplace_intervals": (_i, [_vp, _vp, _vp, _vp, _i, _i64, _vp, _f, _i, _vp]),
    "pcgc_laplace_cdf": (_i, [_vp, _vp, _vp, _i, _i64, _vp, _f, _i, _vp, _vp]),
    "pcgc_debug_quantize_pmf": (_i, [_vp, _vp, _i64, _i, _i, _vp]),
    "pcgc_topk_select": (_i, [_vp, _vp, _i, _i64, _vp, _vp, _vp, _vp]),
    "pcgc_threshold_select": (_i, [_vp, _vp, _i, _i64, _f, _vp, _vp]),
    "pcgc_pmf_to_quantized_cdf": (_i, [_vp, _i64, _i, _i, _vp]),
    "pcgc_range_encode": (_i, [_vp, _i64, _vp, _i, _i, _i, _vp, _i64, C.POINTER(_i64)]),
    "pcgc_range_decode": (_i, [_vp, _i64, _i64, _vp, _i, _i, _i, _vp]),
    "pcgc_range_encode_intervals": (_i, [_vp, _i64, _i, _vp, _i64, C.POINTER(_i64)]),
    "pcgc_range_decode_progress": (_i, [_vp, _i64, _i64, _vp, _i, _i, _i, _vp, _vp, _i64]),
    "pcgc_range_decode_rows": (_i, [_vp, _i64, _i64, _vp, _i, _i, _vp]),
    "pcgc_range_encode_intervals_batch": (_i, [_vp, _i, _i64, _i, _vp, _i64, _vp, _i]),
    "pcgc_range_decode_rows_batch": (_i, [_vp, _vp, _i, _i64, _vp, _vp, _vp, _i, _vp, _i]),
    "pcgc_range_decode_rows_batch_f32": (_i, [_vp, _vp, _i, _i64, _vp, _vp, _vp, _i, _vp, _i]),
    "pcgc_set_deferred_checks": (_i, [_vp, _i]),
    "pcgc_set_quantize_mode": (_i, [_vp, _i, C.c_uint64]),
    "pcgc_debug_noise": (_i, [C.c_uint64, C.c_uint64, _vp]),
    "pcgc_laplace_cdf_dev": (_i, [_vp, _vp, _vp, _i, _i64, _vp, _vp, C.c_double, _f, _i, _vp]),
    "pcgc_range_encode_intervals_dev": (_i, [_vp, _vp, _i, _i64, _i, _vp, _i64, _vp, _vp, _i64, _vp]),
    "pcgc_range_decode_rows_dev": (_i, [_vp, _vp, _vp, _i, _i64, _vp, _vp, C.c_double, _vp, _i, _i, _vp]),
    "pcgc_host_laplace_cdf": (_i, [_vp, _vp, _i, _i64, _vp, _f, _i, _vp, _vp, _i]),
    "pcgc_factorized_cdf_host": (_i, [_vp, _i, _i, _i, _f, _i, _vp]),
    "pcgc_train_conv_forward": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _i, _vp]),
    "pcgc_train_conv_dgrad": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    "pcgc_train_conv_wgrad": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    "pcgc_debug_train_wgrad": (_i, [_vp, _i, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, C.POINTER(_i64)]),
    "pcgc_train_relu_backward": (_i, [_vp, _vp, _vp, _i64, _vp]),
    "pcgc_train_vrn_merge": (_i, [_vp, _vp, _vp, _vp, _i64, _i, _vp]),
    "pcgc_train_vrn_merge_backward": (_i, [_vp, _vp, _vp, _i64, _i, _vp, _vp, _vp]),
    "pcgc_train_abs_floor": (_i, [_vp, _vp, _i64, _f, _vp]),
    "pcgc_train_abs_floor_backward": (_i, [_vp, _vp, _vp, _i64, _f, _vp]),
    "pcgc_train_laplace_backward": (_i, [_vp, _vp, _vp, _vp, _i64, _f, _f, _vp, _vp, _vp]),
    "pcgc_train_factorized_forward": (_i, [_vp, _vp, _vp, _vp, _i, _vp, _i64, C.c_uint64, _f, _vp, _vp]),
    "pcgc_train_factorized_backward": (_i, [_vp, _vp, _vp, _vp, _i, _vp, _i64, _f, _f, _vp, _vp, _vp, _vp]),
    "pcgc_train_bce": (_i, [_vp, _vp, _vp, _i64, _vp]),
    "pcgc_train_bce_backward": (_i, [_vp, _vp, _vp, _i64, _vp, _f, _f, _vp]),
    "pcgc_train_focal": (_i, [_vp, _vp, _vp, _i64, _f, _f, _vp]),
    "pcgc_train_focal_backward": (_i, [_vp, _vp, _vp, _i64, _f, _f, _f, _vp]),
    "pcgc_train_adam": (_i, [_vp, _vp, _vp, _vp, _vp, _i64, _f, _f, _f, _f]),
    "pcgc_host_copy": (_i, [_vp, _vp, _i64, _i]),
    "pcgc_ply_parse": (_i, [_vp, _i64, _vp, _i64, _vp, _i]),
    "pcgc_ply_format": (_i, [_vp, _i64, _vp, _i64, _vp, _i]),
    "pcgc_partition_points": (_i, [_vp, _i64, _i, _i, _vp, _i64, _vp, _vp, _vp, _vp, _vp]),
    "pcgc_voxelize": (_i, [_vp, _vp, _vp, _i, _i, _vp]),
    "pcgc_extract_points": (_i, [_vp, _vp, _i, _i, _vp, _vp, _i64, _vp]),
    "pcgc_geometry_sums": (_i, [_vp, _vp, _i64, _vp, _i64, _vp, _vp]),
    "pcgc_estimate_normals": (_i, [_vp, _vp, _i64, _i, _vp, _vp]),
    "pcgc_mesh_parse": (_i, [_vp, _i64, _i, _vp, _i64, _vp, _i64, C.POINTER(_i64), C.POINTER(_i64)]),
    "pcgc_mesh_sample": (_i, [_vp, _vp, _i64, _vp, _i64, _vp, _i64, C.c_uint64, _i, _vp, C.POINTER(_i64), _vp, _vp]),
}

_lib: Optional[C.CDLL] = None


def lib() -> C.CDLL:
    """Load the shared library (built by ``python -m pcgcv1_b200.build``).  Fails loudly."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "%s is missing: build it with `python -m pcgcv1_b200.build` (there is no CPU fallback)" % LIB_PATH)
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        if l.pcgc_abi_version() != 1:
            raise RuntimeError("libpcgc_b200.so ABI version mismatch")
        _lib = l
    return _lib


class PcgcError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__("pcgc_b200 error %s (%d): %s" % (ERR_NAMES.get(code, "?"), code, msg))
        self.code = code


def check(code: int, ctx=None) -> None:
    if code != 0:
        msg = ""
        if ctx:
            msg = (lib().pcgc_last_error(ctx) or b"").decode("utf-8", "replace")
        raise PcgcError(code, msg)

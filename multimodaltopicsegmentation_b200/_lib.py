"""ctypes binding of libmts_b200.so (the C ABI declared in include/mts_b200.h).

There is no CPU fallback: if the shared library is missing, or a call returns non-zero, this raises.
Build the library with `python -c "import __graft_entry__ as g; g.build()"` or
`make -C multimodaltopicsegmentation_b200/csrc`.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_float, c_int, c_int64, c_uint64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmts_b200.so")
CSRC = os.path.join(_HERE, "csrc")

_P = c_void_p  # every device pointer crosses the ABI as a plain address

# name -> (restype, argtypes); kept in one table so tests can check it against the header
SIGNATURES = {
    "mts_version": (c_int, []),
    "mts_last_error": (ctypes.c_char_p, []),
    "mts_device_ok": (c_int, []),
    "mts_pack_rows_split": (c_int, [_P, c_int64, c_int, _P, c_int64, c_int, c_int, c_int, c_int, _P, _P, _P]),
    "mts_split_tf32": (c_int, [_P, c_int64, c_int, c_int, c_int, c_int, _P, _P, _P]),
    "mts_transpose_split": (c_int, [_P, c_int64, c_int64, c_int, c_int, c_int, c_int, _P, c_int, c_int, _P, _P, _P]),
    "mts_gather_pad": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_float, _P, _P]),
    "mts_gemm_tf32x3": (c_int, [_P, _P, _P, _P, _P, _P, c_int, c_int, c_int, c_int64, c_int, c_int, _P]),
    "mts_gemm_f32": (c_int, [_P, c_int64, _P, c_int64, _P, _P, c_int64, c_int, c_int, c_int, c_int, c_int, c_int,
                             c_int, c_int, c_int, _P, _P]),
    "mts_colsum_ws_bytes": (c_int64, [c_int, c_int]),
    "mts_colsum": (c_int, [_P, c_int64, c_int, c_int, _P, c_int, _P, _P]),
    "mts_lstm_rec_fwd": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, _P, _P, _P]),
    "mts_lstm_rec_fwd_tc": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, _P, _P, _P, _P]),
    "mts_lstm_rec_fwd_tc_bf16": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, _P, _P, _P, _P]),
    "mts_lstm_rec_fwd_tf32": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, _P, _P, _P, _P]),
    "mts_lstm_rec_fwd_h3": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, _P, _P, _P, c_int, _P]),
    "mts_gemm_tf32x3_srcs": (c_int, [_P, c_int, c_int64, _P, c_int, c_int64, _P, _P, _P, _P, _P, c_int, c_int, c_int, c_int64, c_int,
                                     c_int, _P]),
    "mts_pack_rows_f16": (c_int, [_P, c_int64, c_int, _P, c_int64, c_int, c_int, c_int, c_int, _P, _P, _P]),
    "mts_gemm_f16x3": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_int, c_int, c_int, c_int64, c_int, _P]),
    "mts_gemm_tf32x3_gelu_pair": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_int, c_int, c_int, _P]),
    "mts_gemm_bf16p": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int64, c_int, c_int, _P]),
    "mts_gemm_bf16p_out16": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int64, _P]),
    "mts_gemm_bf16p_gelu_pair": (c_int, [_P, _P, _P, _P, _P, c_int, c_int, c_int, _P]),
    "mts_embed_ln_fwd_bf16in": (c_int, [_P, c_int64, _P, _P, _P, _P, c_int, c_int, c_int, c_float, _P, _P, c_int, _P, _P, _P]),
    "mts_band_attn_fwd_bf16": (c_int, [_P, c_int64, c_int64, _P, _P, c_int, c_int, c_int, c_int, c_int, _P, _P, c_int, _P, _P]),
    "mts_band_attn_bf16_supported": (c_int, [c_int]),
    "mts_pack_rows_bf16in": (c_int, [_P, c_int64, c_int, _P, c_int64, c_int, c_int, c_int, c_int, _P, _P]),
    "mts_debug_rec_profile": (c_int, [_P]),
    "mts_debug_rec_profile_h3": (c_int, [_P]),
    "mts_lstm_rec_fwd_h3p": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, _P, _P, _P, c_int, _P]),
    "mts_debug_rec_profile_h3p": (c_int, [_P]),
    "mts_lstm_rec_bwd": (c_int, [_P, _P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, _P, _P]),
    "mts_lstm_rec_bwd_tc": (c_int, [_P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, _P, _P]),
    "mts_lstm_rec_bwd_h3": (c_int, [_P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, _P, _P]),
    "mts_lstm_rec_bwd_tf32": (c_int, [_P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, _P, _P]),
    "mts_head_fwd": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, c_float, _P, _P, _P]),
    "mts_head_bwd_ws_bytes": (c_int64, [c_int, c_int, c_int, c_int]),
    "mts_head_bwd": (c_int, [_P, _P, _P, c_int, c_int, c_int, c_int, _P, _P, _P, _P, _P]),
    "mts_seg_loss_fwd": (c_int, [_P, _P, c_int64, _P, c_int, c_int, c_int, c_float, c_float, c_float, _P, _P, _P]),
    "mts_seg_loss_bwd": (c_int, [_P, _P, c_int64, _P, c_int, c_int, c_int, c_float, c_float, c_float, _P, _P, _P, _P]),
    "mts_seg_metrics": (c_int, [_P, c_int64, _P, c_int64, _P, c_int, c_int, c_int, _P, _P]),
    "mts_crf_viterbi": (c_int, [_P, _P, _P, c_int, c_int, c_int, _P, _P, _P, _P]),
    "mts_crf_nll_fwd": (c_int, [_P, _P, c_int64, _P, _P, c_int, c_int, c_int, _P, _P, _P, _P]),
    "mts_crf_nll_bwd": (c_int, [_P, _P, c_int64, _P, _P, _P, c_int, c_int, c_int, _P, _P, _P, _P]),
    "mts_embed_ln_fwd": (c_int, [_P, c_int64, _P, _P, _P, _P, c_int, c_int, c_int, c_float, _P, _P, _P, c_int, _P, _P, _P, _P,
                                 _P]),
    "mts_embed_ln_fwd_f16": (c_int, [_P, c_int64, _P, _P, _P, _P, c_int, c_int, c_int, c_float, _P, _P, c_int, _P, _P, _P, _P]),
    "mts_add_ln_fwd_f16": (c_int, [_P, _P, _P, _P, c_int, c_int, c_float, _P, _P, c_int, _P, _P]),
    "mts_embed_ln_fwd_pair": (c_int, [_P, c_int64, c_int, _P, c_int64, c_int, _P, _P, _P, _P, c_int, c_int, c_float, _P, _P, _P, c_int,
                                      _P, _P, _P, _P, _P]),
    "mts_embed_ln_fwd_f16_pair": (c_int, [_P, c_int64, c_int, _P, c_int64, c_int, _P, _P, _P, _P, c_int, c_int, c_float, _P, _P, c_int,
                                          _P, _P, _P, _P]),
    "mts_embed_ln_fwd_bf16in_pair": (c_int, [_P, c_int64, c_int, _P, c_int64, c_int, _P, _P, _P, _P, c_int, c_int, c_float, _P, _P,
                                             c_int, _P, _P, _P]),
    "mts_add_ln_fwd": (c_int, [_P, _P, _P, _P, c_int, c_int, c_float, _P, _P, _P, c_int, _P, _P, _P]),
    "mts_gelu_split": (c_int, [_P, c_int64, c_int, c_int, c_int, _P, _P, _P, _P]),
    "mts_band_attn_fwd": (c_int, [_P, c_int64, _P, _P, c_int, c_int, c_int, c_int, c_int, _P, _P, _P, c_int, _P, _P]),
    "mts_band_attn_fwd_mma": (c_int, [_P, c_int64, _P, _P, c_int, c_int, c_int, c_int, c_int, _P, _P, _P, c_int, _P, _P]),
    "mts_band_attn_fwd_simt": (c_int, [_P, c_int64, _P, _P, c_int, c_int, c_int, c_int, c_int, _P, _P, _P, c_int, _P, _P]),
    "mts_band_attn_fwd_tc": (c_int, [_P, c_int64, _P, _P, c_int, c_int, c_int, c_int, c_int, _P, _P, _P, c_int, _P, _P]),
    "mts_band_attn_tc_supported": (c_int, [c_int]),
    "mts_debug_attn_profile": (c_int, [_P]),
    "mts_ln_bwd_ws_bytes": (c_int64, [c_int, c_int]),
    "mts_ln_bwd": (c_int, [_P, _P, _P, _P, c_int, c_int, _P, _P, _P, c_int, _P, _P, _P, _P]),
    "mts_gelu_bwd": (c_int, [_P, _P, c_int, c_int, c_int, _P, _P, _P, _P]),
    "mts_ragged_copy": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, c_float, _P]),
    "mts_embed_bwd": (c_int, [_P, c_int, c_int, c_int, _P, _P, _P, _P]),
    "mts_band_attn_bwd": (c_int, [_P, c_int64, _P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, _P, _P, _P]),
    "mts_band_attn_fwd_dropout": (c_int, [_P, c_int64, _P, _P, c_int, c_int, c_int, c_int, c_int, _P, _P, _P, c_int, _P, c_float,
                                          c_uint64, _P]),
    "mts_band_attn_bwd_dropout": (c_int, [_P, c_int64, _P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, _P, _P, c_float,
                                          c_uint64, _P]),
}

_lib = None


class MtsError(RuntimeError):
    pass


def load():
    """Load libmts_b200.so once; raise loudly if it has not been built (no fallback path exists)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise MtsError(
                f"{LIB_PATH} is missing: the CUDA extension has not been built. Run __graft_entry__.build() "
                "(nvcc -gencode arch=compute_100a,code=sm_100a). There is no CPU fallback.")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name, None)
            if fn is None:
                continue  # declared for a later round; tests/test_abi.py checks header <-> exports
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


_FN = {}


def call(name, *args):
    """Invoke an int-returning entry point and turn a non-zero status into an exception."""
    fn = _FN.get(name)
    if fn is None:
        fn = _FN[name] = getattr(load(), name)
    rc = fn(*args)
    if rc != 0:
        msg = load().mts_last_error().decode("utf-8", "replace")
        raise MtsError(f"{name} failed with status {rc}: {msg}")
    return rc

"""ctypes binding of ``libmodaltune_b200.so`` (the C ABI declared in ``include/modaltune_b200.h``).

The library is built in-tree by ``python -m modaltune_b200.build`` (nvcc, sm_100a).  There is no fallback: if the shared
object is missing or a symbol cannot be resolved, importing the compute path raises.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_float, c_int, c_int32, c_int64, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MODALTUNE_B200_LIB") or os.path.join(HERE, "libmodaltune_b200.so")  # env: experiment builds

MT_F32 = 0
MT_BF16 = 1
MT_MAX_BRANCHES = 8


class DilatedGeometry(Structure):
    """``mt_dilated_geometry`` (include/modaltune_b200.h)."""

    _fields_ = [
        ("n_tokens", c_int32),
        ("n_heads", c_int32),
        ("head_dim", c_int32),
        ("n_branches", c_int32),
        ("seg_len", c_int32 * MT_MAX_BRANCHES),
        ("ratio", c_int32 * MT_MAX_BRANCHES),
    ]


class Dropout(Structure):
    """``mt_dropout`` (include/modaltune_b200.h): train-mode dropout + DropPath of one residual branch."""

    _fields_ = [("p", c_float), ("seed", c_void_p), ("stream_id", c_int64), ("path_scale", c_void_p)]


class LinearEpilogue(Structure):
    """``mt_linear_epilogue`` (include/modaltune_b200.h): what the tensor-core GEMM does with its accumulator."""

    _fields_ = [("mode", c_int32), ("ln_cols", c_int32), ("ln_eps", c_float), ("impl", c_int32),
                ("bias", c_void_p), ("residual", c_void_p), ("col_c1", c_void_p), ("col_c2", c_void_p),
                ("stats", c_void_p), ("ln_mean_out", c_void_p), ("ln_rstd_out", c_void_p), ("out_f32", c_void_p), ("out_bf16", c_void_p),
                ("ld_out_f32", c_int64), ("ld_out_bf16", c_int64), ("ld_residual", c_int64),
                ("out_aux_bf16", c_void_p), ("in_u_bf16", c_void_p), ("in_g_bf16", c_void_p)]


MT_EPI_PLAIN, MT_EPI_GELU_STATS, MT_EPI_LN_RESIDUAL, MT_EPI_GELU_LN_BWD = 0, 3, 4, 5

_G = POINTER(DilatedGeometry)
_D = POINTER(Dropout)
_P = c_void_p
_I64 = c_int64

# name -> (restype, argtypes); mirrors include/modaltune_b200.h one to one (tests/test_abi.py checks the header)
SIGNATURES = {
    "mt_last_error": (c_char_p, []),
    "mt_version": (c_int, []),
    "mt_device_is_sm100": (c_int, []),
    "mt_embed_assemble": (c_int, [_P, c_int, _P, _P, _P, _P, _P, _I64, _I64, _I64, c_float, _P]),
    "mt_layernorm_fwd": (c_int, [_P, c_int, _P, _P, _P, c_int, _I64, _P, c_int, _P, _P, _I64, _I64, c_float, _P]),
    "mt_layernorm_bwd": (c_int, [_P, c_int, _P, c_int, _P, _P, _P, _P, c_int, _P, c_int, _P, _P, _P, _I64, _I64, _P]),
    "mt_layernorm_bwd_ws": (c_int, [_P, c_int, _P, c_int, _P, _P, _P, _P, c_int, _P, c_int, _P, _P, _P, _I64, _I64, _P, _I64,
                                    _P]),
    "mt_colreduce_workspace_floats": (_I64, [_I64]),
    "mt_layernorm_bwd_ffn_prep": (c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I64, _I64, _I64, _P]),
    "mt_add_layernorm_fwd": (c_int, [_P, _P, c_int, _P, _P, _P, _P, _P, c_int, _P, _P, _I64, _I64, c_float, _D, _P]),
    "mt_gelu_ln_fwd": (c_int, [_P, c_int, _P, _P, _P, _P, c_int, _P, _P, _I64, _I64, c_float, _P]),
    "mt_gelu_ln_bwd": (c_int, [_P, c_int, _P, c_int, _P, _P, _P, _P, _P, c_int, _I64, _I64, _P]),
    "mt_linear_sm100": (c_int, [_P, _I64, _P, _I64, _I64, _I64, _I64, POINTER(LinearEpilogue), _P]),
    "mt_ffn_bwd_prep": (c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _I64, _I64, _I64, _P]),
    "mt_dilated_attn_fwd": (c_int, [_G, _P, _I64, _I64, c_int, _P, _P, c_int, _P]),
    "mt_dilated_attn_fwd_batch": (c_int, [_G, _P, _I64, _I64, c_int, c_int, _P, _P, c_int, _P]),
    "mt_dilated_merge_ln_fwd": (c_int, [_G, _P, _P, c_int, _P, _P, _P, _P, c_float, _P, _P, _P, _P]),
    "mt_dilated_merge_ln_bwd": (c_int, [_G, _P, c_int, _P, _P, _P, _P, _P, c_int, _P, _P, _P]),
    "mt_dilated_attn_bwd": (c_int, [_G, _P, _I64, _I64, _P, _P, _P, c_int, _P, c_int, _P]),
    "mt_cross_attn_fwd": (c_int, [_P, _I64, _P, _P, _I64, c_int, _P, _I64, _P, _I64, _I64, c_int, c_int, _P, _I64, c_int, _P]),
    "mt_cross_attn_bwd": (c_int, [_P, _I64, _P, _P, _I64, _P, _P, _I64, _P, c_int, _P, _I64, _P, _P, _I64, _I64, _I64, c_int,
                                  c_int, c_int, _P]),
    "mt_cross_attn_workspace_floats": (_I64, [_I64, _I64, c_int, c_int, c_int, c_int]),
    "mt_cross_attn_bwd_ws": (c_int, [_P, _I64, _P, _P, _I64, _P, _P, _I64, _P, c_int, _P, _I64, _P, _P, _I64, _I64, _I64,
                                     c_int, c_int, _P, _I64, c_int, _P]),
    "mt_cross_attn_bwd_workspace_floats": (_I64, [_I64, _I64, c_int, c_int, c_int, c_int]),
    "mt_cross_attn_probs": (c_int, [_P, _I64, _P, _I64, c_int, _P, _P, _I64, _I64, _I64, c_int, c_int, c_int, _P]),
    "mt_gated_residual": (c_int, [_P, _P, c_int, _P, _P, _I64, _I64, _P]),
    "mt_gated_residual_bwd": (c_int, [_P, _P, _P, c_int, _P, _P, _P, c_int, _P, _P, _I64, _I64, _P]),
    "mt_gated_residual_bwd_ws": (c_int, [_P, _P, _P, c_int, _P, _P, _P, c_int, _P, _P, _I64, _I64, _P, _I64, _P]),
    "mt_residual_bias_add": (c_int, [_P, _P, c_int, _P, _P, _I64, _I64, _D, _P]),
    "mt_dropout_bwd_cast": (c_int, [_P, c_int, _P, c_int, _I64, _D, _P]),
    "mt_cast": (c_int, [_P, c_int, _P, c_int, _I64, _P]),
    "mt_colsum": (c_int, [_P, _I64, _P, _I64, _I64, _P]),
    "mt_colsum_ws": (c_int, [_P, _I64, _P, _I64, _I64, _P, _I64, _P]),
}

_lib = None


def load() -> ctypes.CDLL:
    """Load the shared library and bind every entry point; raises if it is absent (no CPU fallback exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -m modaltune_b200.build` (nvcc, sm_100a). "
            "modaltune_b200 has no CPU or PyTorch fallback for its kernels.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error() -> str:
    return load().mt_last_error().decode("utf-8", "replace")

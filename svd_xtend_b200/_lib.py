"""ctypes binding of the C ABI in include/svd_xtend_b200.h.

The product path has no CPU fallback: if the shared library is missing or fails to load,
importing any op raises. (It is built in-tree by ``svd_xtend_b200.build`` /
``__graft_entry__.build`` and travels to the GPU box with the repo snapshot.)
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

PKG = Path(__file__).resolve().parent
# SVDX_LIB selects an alternative build of the same library (kernel tuning experiments: svd_xtend_b200.build.build_variant)
LIB_PATH = Path(os.environ["SVDX_LIB"]) if os.environ.get("SVDX_LIB") else PKG / "lib" / "libsvdx_b200.so"

SVDX_MAX_TAPS = 27
A_ROWS, A_CONV2D = 0, 1
OUT_BF16, OUT_F32, OUT_F32_ATOMIC = 0, 1, 2
ACT_NONE, ACT_GELU = 0, 1
SVDX_CLIP_MAX_TAPS = 31

c_void_p, c_int, c_i64, c_float = C.c_void_p, C.c_int32, C.c_int64, C.c_float


class SvdxTapGemm(C.Structure):
    _fields_ = [
        ("a", c_void_p), ("lda", c_i64), ("a_mode", c_int), ("a_major_mn", c_int),
        ("rows_per_group", c_int), ("groups", c_int),
        ("W", c_int), ("H", c_int), ("nimg", c_int),
        ("num_taps", c_int),
        ("tap_d0", c_int * SVDX_MAX_TAPS), ("tap_d1", c_int * SVDX_MAX_TAPS), ("tap_d2", c_int * SVDX_MAX_TAPS),
        ("b", c_void_p), ("ldb", c_i64), ("b_major_mn", c_int), ("b_mode", c_int),
        ("M", c_int), ("N", c_int), ("K", c_int),
        ("block_n", c_int), ("split_k", c_int),
        ("out", c_void_p), ("ldo", c_i64), ("out_dtype", c_int), ("geglu", c_int),
        ("bias", c_void_p), ("rowbias", c_void_p), ("rowbias_div", c_int), ("ldrb", c_i64),
        ("res1", c_void_p), ("ldr1", c_i64), ("res2", c_void_p), ("ldr2", c_i64),
        ("scales", c_void_p), ("pre", c_void_p), ("ldpre", c_i64),
        ("gn_sum", c_void_p), ("gn_ld", c_i64), ("gn_rows", c_int),
        ("gnb_x", c_void_p), ("gnb_ldx", c_i64), ("gnb_x2", c_void_p), ("gnb_ldx2", c_i64), ("gnb_c1", c_int),
        ("gnb_ab", c_void_p), ("gnb_sum", c_void_p), ("gnb_rows", c_int), ("gnb_silu", c_int),
        ("act", c_int),
    ]


class SvdxAttn(C.Structure):
    _fields_ = [
        ("q", c_void_p), ("k", c_void_p), ("v", c_void_p), ("o", c_void_p),
        ("ldq", c_i64), ("ldk", c_i64), ("ldv", c_i64), ("ldo", c_i64),
        ("nseq", c_int), ("heads", c_int), ("S", c_int), ("inner", c_int),
        ("outer_stride", c_i64), ("inner_stride", c_i64), ("tok_stride", c_i64),
        ("scale", c_float), ("lse", c_void_p),
        ("dout", c_void_p), ("lddo", c_i64),
        ("dq", c_void_p), ("dk", c_void_p), ("dv", c_void_p),
        ("lddq", c_i64), ("lddk", c_i64), ("lddv", c_i64),
        ("delta", c_void_p),
    ]


class SvdxClipPixels(C.Structure):
    _fields_ = [
        ("x", c_void_p), ("dtype", c_int), ("B", c_int), ("H", c_int), ("W", c_int), ("resize", c_int),
        ("ky", c_int), ("kx", c_int),
        ("wy", C.c_double * SVDX_CLIP_MAX_TAPS), ("wx", C.c_double * SVDX_CLIP_MAX_TAPS),
        ("mean", C.c_double * 3), ("std", C.c_double * 3),
        ("out", c_void_p), ("ldo", c_i64),
    ]


_PROTOS = {
    "svdx_tapgemm": [C.POINTER(SvdxTapGemm), c_void_p],
    "svdx_splitk_epilogue": [c_void_p, c_i64, c_void_p, c_i64, c_i64, c_int, c_void_p, c_void_p, c_int, c_i64, c_void_p, c_i64,
                             c_void_p, c_i64, c_void_p, c_void_p],
    "svdx_splitk_epilogue_act": [c_void_p, c_i64, c_void_p, c_i64, c_i64, c_int, c_void_p, c_void_p, c_int, c_i64, c_void_p, c_i64,
                                 c_void_p, c_i64, c_void_p, c_int, c_void_p],
    "svdx_num_sms": [],
    "svdx_enable_peer_access": [c_int],
    "svdx_ipc_export": [c_void_p, c_void_p, c_void_p],
    "svdx_ipc_import": [c_void_p, c_i64, c_void_p],
    "svdx_struct_size": [c_int],
    "svdx_groupnorm_stats": [c_void_p, c_i64, c_int, c_void_p, c_i64, c_int, c_int, c_int, c_int, c_float,
                             c_void_p, c_void_p, c_void_p],
    "svdx_groupnorm_apply": [c_void_p, c_i64, c_int, c_void_p, c_i64, c_int, c_int, c_int, c_int,
                             c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_i64, c_void_p, c_void_p],
    "svdx_groupnorm_apply_fused": [c_void_p, c_i64, c_int, c_void_p, c_i64, c_int, c_int, c_int, c_int, c_float,
                                   c_void_p, c_i64, c_void_p, c_i64, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_i64, c_void_p,
                                   c_void_p],
    "svdx_groupnorm_bwd_fused": [c_void_p, c_i64, c_int, c_void_p, c_i64, c_int, c_void_p, c_i64, c_int, c_int, c_int,
                                 c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_i64, c_void_p, c_i64,
                                 c_void_p, c_void_p, c_void_p, c_i64, c_void_p],
    "svdx_groupnorm_bwd": [c_void_p, c_i64, c_int, c_void_p, c_i64, c_int, c_void_p, c_i64, c_int, c_int, c_int,
                           c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_i64, c_void_p, c_i64,
                           c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_i64, c_void_p],
    "svdx_layernorm_fwd": [c_void_p, c_i64, c_int, c_int, c_void_p, c_void_p, c_float, c_void_p, c_i64,
                           c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_i64, c_void_p],
    "svdx_layernorm_bwd": [c_void_p, c_i64, c_void_p, c_i64, c_int, c_int, c_void_p, c_void_p, c_void_p,
                           c_void_p, c_i64, c_void_p, c_i64, c_void_p, c_void_p, c_void_p],
    "svdx_attention_fwd": [C.POINTER(SvdxAttn), c_void_p],
    "svdx_attention_bwd": [C.POINTER(SvdxAttn), c_void_p],
    "svdx_attention_vit_fwd": [C.POINTER(SvdxAttn), c_void_p],
    "svdx_clip_pixels": [C.POINTER(SvdxClipPixels), c_void_p],
    "svdx_prep_weight": [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p],
    "svdx_unprep_conv_grad": [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p],
    "svdx_dot_diff": [c_void_p, c_void_p, c_void_p, c_i64, c_void_p, c_void_p],
    "svdx_silu_bwd_f32": [c_void_p, c_void_p, c_void_p, c_i64, c_void_p],
    "svdx_cast_f32_bf16": [c_void_p, c_void_p, c_i64, c_void_p],
    "svdx_cast_bf16_f32": [c_void_p, c_void_p, c_i64, c_void_p],
    "svdx_cast_f16_f32": [c_void_p, c_void_p, c_i64, c_void_p],
    "svdx_nchw_to_nhwc": [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p],
    "svdx_nhwc_to_nchw": [c_void_p, c_i64, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p],
    "svdx_upsample2x": [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p],
    "svdx_upsample2x_bwd": [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p],
    "svdx_space_to_planes": [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p],
    "svdx_planes_to_space": [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p],
    "svdx_concat_channels": [c_void_p, c_int, c_void_p, c_int, c_void_p, c_i64, c_void_p],
    "svdx_split_channels": [c_void_p, c_void_p, c_int, c_void_p, c_int, c_i64, c_int, c_void_p],
    "svdx_add_bf16": [c_void_p, c_void_p, c_void_p, c_i64, c_void_p],
    "svdx_axpby_bf16": [c_void_p, c_void_p, c_void_p, c_void_p, c_i64, c_void_p],
    "svdx_silu_f32": [c_void_p, c_void_p, c_i64, c_void_p],
    "svdx_colsum": [c_void_p, c_i64, c_i64, c_int, c_void_p, c_int, c_void_p],
    "svdx_geglu_bwd": [c_void_p, c_i64, c_void_p, c_i64, c_void_p, c_i64, c_i64, c_int, c_void_p, c_void_p],
    "svdx_softmax_rows": [c_void_p, c_i64, c_i64, c_int, c_float, c_void_p, c_i64, c_void_p],
    "svdx_gemv": [c_void_p, c_i64, c_void_p, c_i64, c_int, c_int, c_int, c_void_p, c_void_p, c_i64, c_int, c_float, c_int, c_void_p],
    "svdx_outer_accum": [c_void_p, c_i64, c_void_p, c_i64, c_int, c_int, c_int, c_void_p, c_void_p, c_i64, c_void_p],
    "svdx_blend_scales": [c_void_p, c_void_p, c_void_p],
    "svdx_adamw": [c_void_p, c_void_p, c_void_p, c_void_p, c_i64, c_float, c_float, c_float, c_float, c_float,
                   c_int, c_float, c_void_p, c_void_p],
    "svdx_adamw_graph": [c_void_p, c_void_p, c_void_p, c_void_p, c_i64, c_void_p, c_float, c_void_p, c_void_p],
    "svdx_adamw_p2p": [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_i64, c_i64, c_void_p, c_float, c_int, c_void_p],
    "svdx_multi_transpose": [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p],
}

EXPORTED_SYMBOLS = tuple(_PROTOS) + ("svdx_last_error",)

_lib = None


def load() -> C.CDLL:
    """Load the C-ABI library; raises (never falls back) when it is missing."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise RuntimeError(
                f"svd_xtend_b200: native library {LIB_PATH} is missing — run `python -m svd_xtend_b200.build` "
                "(there is no CPU or PyTorch fallback for the hot path)")
        lib = C.CDLL(str(LIB_PATH))
        missing = [n for n in _PROTOS if not hasattr(lib, n)]
        if missing and os.environ.get("SVDX_ALLOW_PARTIAL"):  # kernel bring-up only
            for n in missing:
                _PROTOS.pop(n)
            missing = []
        if missing:
            raise RuntimeError(f"svd_xtend_b200: {LIB_PATH} lacks symbols {missing}; rebuild it")
        for name, args in _PROTOS.items():
            fn = getattr(lib, name)
            fn.argtypes = args
            fn.restype = C.c_int
        if (lib.svdx_struct_size(0) != C.sizeof(SvdxTapGemm) or lib.svdx_struct_size(1) != C.sizeof(SvdxAttn)
                or lib.svdx_struct_size(2) != C.sizeof(SvdxClipPixels)):
            raise RuntimeError("svd_xtend_b200: ctypes struct layout does not match the C ABI")
        lib.svdx_last_error.restype = C.c_char_p
        lib.svdx_last_error.argtypes = []
        _lib = lib
    return _lib


class SvdxError(RuntimeError):
    pass


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().svdx_last_error().decode(errors="replace")
        raise SvdxError(f"{what} failed with status {rc}: {msg}")

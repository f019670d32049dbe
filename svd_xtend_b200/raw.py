"""Thin tensor-level wrappers over the C ABI (no autograd): pointer/shape marshalling only."""
from __future__ import annotations

import ctypes as C
import functools
import math
import os
from typing import Optional, Sequence

import torch

from . import _lib
from ._lib import A_CONV2D, A_ROWS, ACT_GELU, ACT_NONE, OUT_BF16, OUT_F32, OUT_F32_ATOMIC, SvdxAttn, SvdxClipPixels, SvdxTapGemm, load

bf16 = torch.bfloat16

# source-dtype codes of the C ABI (include/svd_xtend_b200.h, "elementwise / layout")
_DTYPE_CODE = {torch.float32: 0, torch.bfloat16: 1, torch.float16: 2}


def dtype_code(t: torch.Tensor, what: str) -> int:
    """dtype code of a parameter / boundary tensor; anything but fp32 / bf16 / fp16 is rejected loudly (a silently
    misread buffer would be an out-of-bounds read)."""
    try:
        return _DTYPE_CODE[t.dtype]
    except KeyError:
        raise TypeError(f"svd_xtend_b200: {what} has dtype {t.dtype}; supported: float32, bfloat16, float16") from None

# number of kernels launched through the C ABI since import (each wrapper adds what its entry point launches)
LAUNCHES = [0]
_KERNELS_PER_CALL = {"svdx_groupnorm_stats": 2, "svdx_groupnorm_bwd": 2, "svdx_groupnorm_apply_fused": 1, "svdx_attention_bwd": 3, "svdx_adamw_graph": 2, "svdx_adamw_p2p": 2}


def check(rc: int, what: str = "") -> None:
    LAUNCHES[0] += _KERNELS_PER_CALL.get(what, 1)
    _lib.check(rc, what)


# ---- measurement hooks (bench.py): per-family accounting of algorithmic work and in-graph ablation -------------------
# Families: "linear" / "conv" (svdx_tapgemm), "attention", "groupnorm", "layernorm", "adamw", "elementwise".
# ACCOUNT(family, flops, bytes) is called for every launch while set; a family named in ABLATE is NOT launched (its
# outputs stay uninitialised: only for timing a captured step with that family removed, never for results).
ABLATE: set = set()
ACCOUNT = None
SHAPE_LOG = None     # list: one record per svdx_tapgemm launch, in launch order (joined with the ncu launch list by scripts/)


def _fam(family: str, flops: float = 0.0, nbytes: float = 0.0) -> bool:
    if ACCOUNT is not None:
        ACCOUNT(family, flops, nbytes)
    return family in ABLATE


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _rowmajor(t: torch.Tensor, name: str) -> int:
    """leading dimension (elements) of a 2-D-like view whose last dim is contiguous."""
    if t.stride(-1) != 1:
        raise ValueError(f"{name}: last dimension must be contiguous")
    return t.stride(-2)


def pick_block_n(n_out: int, mn_major: bool = False) -> int:
    if mn_major:
        for bn in (256, 192, 128, 64):
            if n_out % bn == 0:
                return bn
        return 256 if n_out > 256 else ((n_out + 63) // 64) * 64
    for bn in (256, 160, 128, 96, 64, 32):
        if n_out % bn == 0:
            return bn
    return 256 if n_out > 256 else ((n_out + 31) // 32) * 32


_NUM_SMS = [0]


def num_sms() -> int:
    if _NUM_SMS[0] == 0:
        _NUM_SMS[0] = int(load().svdx_num_sms())
    return _NUM_SMS[0]


PAIR_MODE = os.environ.get("SVDX_2CTA", "1") != "0"     # mirrors SVDX_2CTA_DEFAULT of tapgemm_common.cuh
_L2_BYTES_PER_CLK = 4500.0                                # ~8.5 TB/s L2->SM at 1.9 GHz (measured, profiles/)


def pair_eligible(M: int, n_out: int, bn_out: int, geglu: bool) -> bool:
    """same rule as svdx_tapgemm2_eligible (tapgemm2.cu) for K-major problems without split-K"""
    bn = 2 * bn_out if geglu else bn_out
    return PAIR_MODE and M >= 512 and bn >= 64 and bn % 32 == 0 and (bn // 2) % 8 == 0 and n_out % bn_out == 0


def _tile_cost(M: int, n_out: int, bn_out: int, geglu: bool, sms: int) -> float:
    """relative time of the whole problem with output tiles 128 x bn_out (256 x bn_out for a CTA pair):
    waves over the SMs x per-k-block time = max(tensor pipe, L2->SM bytes at the measured chip bandwidth)."""
    bn = 2 * bn_out if geglu else bn_out
    m_tiles = (M + 127) // 128
    n_tiles = (n_out + bn_out - 1) // bn_out
    pair = pair_eligible(M, n_out, bn_out, geglu)
    if pair:
        ctas = 2 * ((m_tiles + 1) // 2) * n_tiles
        bytes_kb = 16384 + 64 * bn
    else:
        ctas = m_tiles * n_tiles
        bytes_kb = 16384 + 128 * bn
    active = min(ctas, sms)
    mma = 4 * max(bn / 2.0, 32.0 + bn / 4.0 if not pair else bn / 2.0)
    l2 = bytes_kb * active / _L2_BYTES_PER_CLK
    waves = (ctas + sms - 1) // sms
    return waves * max(mma, l2)


def choose_block_n(M: int, n_out: int, geglu: bool = False, mn_major: bool = False) -> int:
    """tile width for svdx_tapgemm: minimises the modelled time (see _tile_cost) over the widths that tile n_out
    exactly. Small-M levels get narrow tiles that fill the SMs; large-M levels get the widest tile (fewest L2 bytes per
    FLOP). Returns the block_n of the C ABI (2x the output width for GEGLU)."""
    sms = num_sms()
    if mn_major:
        best, best_cost = None, None
        m_tiles = (M + 127) // 128
        for bn in (256, 192, 128, 64):
            cost = m_tiles * ((n_out + bn - 1) // bn) * max(bn / 2.0, 32.0 + bn / 4.0)
            if best_cost is None or cost < best_cost - 1e-9:
                best, best_cost = bn, cost
        return best
    cands = [128, 64, 32] if geglu else [256, 160, 128, 96, 64, 32]
    best, best_cost = None, None
    for bn in cands:
        if n_out % bn and n_out > bn:
            continue
        cost = _tile_cost(M, n_out, bn, geglu, sms)
        if best_cost is None or cost < best_cost * 0.98:
            best, best_cost = bn, cost
    if best is None:
        best = pick_block_n(n_out, False)
    return 2 * best if geglu else best


WIDE_TILE = os.environ.get("SVDX_WIDE", "1") != "0"
WIDE_MIN_K = int(os.environ.get("SVDX_WIDE_MIN_K", "960"))


def _wide_tile_ok(M, N, k_total, out, ldo, geglu, a_mn, b_mn, b_mode, split_k, out_dtype, bias, rowbias) -> bool:
    """256 x 320 CTA-pair tiles (svdx_tapgemm block_n = 320: the A tile crosses L2 once per 320 output columns instead of
    once per 160) for the C = 320 / 640 / 960 layers when the contraction is long enough to hide the partly exposed epilogue
    of the overlapping accumulators. Mirrors the library's conditions for the wide form (CTA-pair kernel, bf16 TMA-store
    epilogues); anything else keeps choose_block_n's width."""
    # measured (scripts/kbench.py gemm, profiles/r2_kbench_gemm.txt): wins 8-25 % where the alternative is 160-wide tiles and
    # K * taps >= 960 (convs at C = 320 / 640: 1.06 -> 1.30-1.43 PFLOP/s); loses against 256-wide tiles (N % 256 == 0) and
    # at short K, where the partly exposed epilogue costs more than the A traffic saved
    if not WIDE_TILE or geglu or a_mn or b_mn or b_mode != 0 or split_k != 1 or N % 320 or N % 256 == 0 or M < 512 or k_total < WIDE_MIN_K:
        return False
    if out.dtype != bf16 or (out_dtype is not None and out_dtype != OUT_BF16):
        return False
    ld = ldo if ldo is not None else out.stride(0)
    if ld % 8 or out.data_ptr() % 16:
        return False
    if bias is not None and bias.data_ptr() % 16:
        return False
    if rowbias is not None and (rowbias.data_ptr() % 16 or rowbias.stride(0) % 4):
        return False
    return True


_WGRAD_L2_BYTES_PER_CLK = 6500.0     # fitted to profiles/r2_kbench.txt (weight-gradient GEMMs are L2 -> SM bound)


def wgrad_plan(O: int, K: int, M: int):
    """(block_n, split_k) of a weight-gradient GEMM dW[O, K] += dy[M, O]^T x[M, K] (MN-major operands, fp32 reduce-add
    epilogue). Tile width and the split of the token contraction are chosen TOGETHER by a small model fitted to measured
    launches (profiles/r2_kbench.txt): CTAs = tiles * split, time = waves * (k-blocks per CTA * max(tensor pipe, L2 -> SM bytes of the
    CTAs running concurrently) + tile reduce-add). The round-1 rule picked the tile width alone from MMA efficiency and
    chose 128-wide tiles at K = 640, twice the L2 traffic of 256-wide ones (100 us vs 62 us for O = 5120, K = 640)."""
    sms = num_sms()
    kb = (M + 63) // 64
    m_tiles = (O + 127) // 128
    best = None
    for bn in ((192, 256, 128) if K > 64 else (64,)):     # ties go to the earlier width
        n_tiles = (K + bn - 1) // bn
        tiles = m_tiles * n_tiles
        splits = {1, max(1, min(kb // 32, sms // max(tiles, 1))), max(1, min(kb // 8, -(-sms // max(tiles, 1))))}
        for split in sorted(splits):
            ctas = tiles * split
            active = min(ctas, sms)
            bytes_kb = 16384 + 128.0 * K / n_tiles            # out-of-range B columns of the last tile are not fetched
            per = max(4.0 * max(bn / 2.0, 32.0 + bn / 4.0), bytes_kb * active / _WGRAD_L2_BYTES_PER_CLK)
            waves = -(-ctas // sms)
            cost = waves * ((kb / split) * per + bn * 8.0 + 3000.0)
            if best is None or cost < best[0] * 0.97:
                best = (cost, bn, split)
    return best[1], best[2]


def tapgemm(
    a: torch.Tensor,
    b: torch.Tensor,
    out: torch.Tensor,
    *,
    M: int,
    N: int,
    K: int,
    mode: int = A_ROWS,
    taps: Sequence[Sequence[int]] = ((0, 0, 0),),
    rows_per_group: Optional[int] = None,
    groups: int = 1,
    conv_whn: Optional[Sequence[int]] = None,
    lda: Optional[int] = None,
    ldb: Optional[int] = None,
    ldo: Optional[int] = None,
    a_mn: bool = False,
    b_mn: bool = False,
    b_mode: int = 0,
    block_n: Optional[int] = None,
    split_k: int = 1,
    out_dtype: Optional[int] = None,
    geglu: bool = False,
    bias: Optional[torch.Tensor] = None,
    rowbias: Optional[torch.Tensor] = None,
    rowbias_div: int = 1,
    res1: Optional[torch.Tensor] = None,
    res2: Optional[torch.Tensor] = None,
    scales: Optional[torch.Tensor] = None,
    pre: Optional[torch.Tensor] = None,
    gn_sum: Optional[torch.Tensor] = None,
    gn_rows: int = 0,
    gnb: Optional[dict] = None,
    act: int = ACT_NONE,
) -> torch.Tensor:
    """Launch svdx_tapgemm on the current stream. All tensors are CUDA; a/b/res/pre are bf16.
    gn_sum: zeroed fp32 [slabs, 2, C] buffer that receives the per-channel sum / sum of squares of the output (fused
    GroupNorm statistics), one slab per gn_rows output rows.
    act: activation of acc + bias + rowbias before the residual step (ACT_GELU: the erf GELU; bf16 output only)."""
    family = "conv" if (mode == A_CONV2D or len(taps) > 1 or b_mode != 0) else "linear"
    if _fam(family, 2.0 * M * N * K * len(taps)):
        return out
    if SHAPE_LOG is not None:
        SHAPE_LOG.append(dict(M=M, N=N, K=K, taps=len(taps), conv2d=int(mode == A_CONV2D), geglu=int(geglu), a_mn=int(a_mn), b_mode=b_mode,
                              split_k=split_k, block_n=block_n, f32out=int(out.dtype != bf16), bias=int(bias is not None),
                              rowbias=int(rowbias is not None), res=int(res1 is not None) + int(res2 is not None),
                              scales=int(scales is not None), pre=int(pre is not None)))
    d = SvdxTapGemm()
    assert a.dtype == bf16 and b.dtype == bf16
    d.a = a.data_ptr()
    d.lda = lda if lda is not None else _rowmajor(a, "a")
    d.a_mode = mode
    d.a_major_mn = int(a_mn)
    d.rows_per_group = rows_per_group if rows_per_group is not None else M
    d.groups = groups
    if conv_whn is not None:
        d.W, d.H, d.nimg = conv_whn
    d.num_taps = len(taps)
    for i, t in enumerate(taps):
        d.tap_d0[i], d.tap_d1[i], d.tap_d2[i] = int(t[0]), int(t[1]), int(t[2])
    d.b = b.data_ptr()
    d.ldb = ldb if ldb is not None else _rowmajor(b, "b")
    d.b_major_mn = int(b_mn)
    d.b_mode = b_mode
    d.M, d.N, d.K = M, N, K
    n_out = N // 2 if geglu else N
    if block_n is None:
        block_n = choose_block_n(M, n_out, geglu, b_mn)
        if _wide_tile_ok(M, N, K * len(taps), out, ldo, geglu, a_mn, b_mn, b_mode, split_k, out_dtype, bias, rowbias):
            block_n = 320
    d.block_n = block_n
    d.split_k = split_k
    d.out = out.data_ptr()
    d.ldo = ldo if ldo is not None else _rowmajor(out, "out")
    if out_dtype is None:
        out_dtype = OUT_BF16 if out.dtype == bf16 else OUT_F32
    d.out_dtype = out_dtype
    d.geglu = int(geglu)
    if bias is not None:
        assert bias.dtype == torch.float32
        d.bias = bias.data_ptr()
    if rowbias is not None:
        assert rowbias.dtype == torch.float32
        d.rowbias = rowbias.data_ptr()
        d.rowbias_div = rowbias_div
        d.ldrb = _rowmajor(rowbias, "rowbias")
    if res1 is not None:
        assert res1.dtype == bf16
        d.res1 = res1.data_ptr()
        d.ldr1 = _rowmajor(res1, "res1")
    if res2 is not None:
        assert res2.dtype == bf16
        d.res2 = res2.data_ptr()
        d.ldr2 = _rowmajor(res2, "res2")
    if scales is not None:
        assert scales.dtype == torch.float32 and scales.numel() >= 3
        d.scales = scales.data_ptr()
    if pre is not None:
        assert pre.dtype == bf16
        d.pre = pre.data_ptr()
        d.ldpre = _rowmajor(pre, "pre")
    if gn_sum is not None:
        assert gn_sum.dtype == torch.float32 and gn_sum.dim() == 3 and gn_sum.shape[1] == 2 and gn_sum.is_contiguous() and gn_rows > 0
        d.gn_sum = gn_sum.data_ptr()
        d.gn_ld = gn_sum.shape[2]
        d.gn_rows = gn_rows
    if gnb is not None:
        # GroupNorm-backward sums of the output (= dL/d(GroupNorm output)): x / x2 the GroupNorm input, ab its forward
        # scale / shift table, sum the zeroed fp32 [slabs, 2, N] accumulator, rows per slab, silu flag
        gx, gx2 = gnb["x"], gnb.get("x2")
        assert gx.dtype == bf16 and gnb["sum"].dtype == torch.float32 and gnb["sum"].is_contiguous() and gnb["sum"].shape[-1] == N
        d.gnb_x = gx.data_ptr()
        d.gnb_ldx = _rowmajor(gx, "gnb x")
        if gx2 is not None:
            d.gnb_x2 = gx2.data_ptr()
            d.gnb_ldx2 = _rowmajor(gx2, "gnb x2")
            d.gnb_c1 = gx.shape[-1]
        d.gnb_ab = _ptr(gnb.get("ab"))
        d.gnb_sum = gnb["sum"].data_ptr()
        d.gnb_rows = gnb["rows"]
        d.gnb_silu = int(gnb["silu"])
    d.act = int(act)
    check(load().svdx_tapgemm(C.byref(d), _stream()), "svdx_tapgemm")
    return out


_SPLITK_WS: dict = {}


def _splitk_workspace(M: int, N: int, device) -> torch.Tensor:
    """one zeroed fp32 [M, N] workspace per shape and device: svdx_splitk_epilogue re-zeroes what it reads, so the
    accumulate -> epilogue pairs of a stream can share it without a memset per launch"""
    # per stream: two streams must never interleave accumulate -> epilogue pairs on one workspace
    key = (M, N, str(device), _stream() if torch.device(device).type == "cuda" else 0)
    ws = _SPLITK_WS.get(key)
    if ws is None:
        ws = torch.zeros(M, N, device=device, dtype=torch.float32)
        _SPLITK_WS[key] = ws
    return ws


def split_plan(out_is_bf16: bool, M: int, N: int, K: int, ntaps: int = 1, geglu=False, a_mn=False, b_mn=False, block_n=None):
    """(tile width, split factor) of the automatic split-K path of tapgemm_auto, or None when the problem is launched whole.
    Small-M / long-K problems whose 128x256 tiles cannot fill the SMs split the contraction over CTAs."""
    if not (out_is_bf16 and not geglu and not a_mn and not b_mn and block_n is None and N % 8 == 0 and N >= 256):
        return None
    bn = 256 if N % 256 == 0 else (160 if N % 160 == 0 else 0)
    if not bn:
        return None
    kb = ((K + 63) // 64) * ntaps
    tiles = ((M + 127) // 128) * (N // bn)
    split = min(num_sms() // max(tiles, 1), kb // 8)
    if tiles <= num_sms() // 3 and split >= 2:
        return bn, split
    return None


def tapgemm_auto(a, b, out, *, M, N, K, taps=((0, 0, 0),), bias=None, rowbias=None, rowbias_div=1, res1=None, res2=None,
                 scales=None, gn_sum=None, gn_rows=0, act=ACT_NONE, **kw):
    """svdx_tapgemm with automatic split-K for small-M / long-K problems (bf16 output, K-major operands, no GEGLU):
    when 128x256 tiles cannot fill the SMs, the contraction is split over CTAs (fp32 atomics into a workspace) and
    svdx_splitk_epilogue(_act) applies bias / row-bias / activation / residuals / scales. Fused GroupNorm statistics (gn_sum)
    exist on the whole-problem path only: callers ask `split_plan` first and keep the stand-alone statistics kernel for split
    outputs."""
    kw = dict(kw)
    if kw.get("block_n") is None:
        kw.pop("block_n", None)
    if (M <= 8 and not act and len(taps) == 1 and kw.get("mode", A_ROWS) == A_ROWS and not kw.get("geglu") and not kw.get("a_mn") and not kw.get("b_mn")
            and rowbias is None and res1 is None and res2 is None and scales is None and gn_sum is None and kw.get("groups", 1) == 1
            and K % 8 == 0 and a.stride(-1) == 1 and b.stride(-1) == 1 and out.dtype in (bf16, torch.float32)):
        # conditioning vectors ([B, C] rows): a GEMV, not a 128-row tensor-core tile
        return gemv(a, b, out, M=M, N=N, K=K, bias=bias, lda=kw.get("lda"), ldw=kw.get("ldb"))
    plan = split_plan(out.dtype == bf16, M, N, K, len(taps), kw.get("geglu"), kw.get("a_mn"), kw.get("b_mn"), kw.get("block_n"))
    if plan is not None:
        assert gn_sum is None, "fused GroupNorm statistics are not available on the split-K path"
        bn, split = plan
        ws = _splitk_workspace(M, N, out.device)
        tapgemm(a, b, ws, M=M, N=N, K=K, taps=taps, block_n=bn, split_k=split, out_dtype=OUT_F32_ATOMIC, **kw)
        if _fam("conv" if (kw.get("mode", A_ROWS) == A_CONV2D or len(taps) > 1) else "linear"):
            return out
        check(load().svdx_splitk_epilogue_act(ws.data_ptr(), N, out.data_ptr(), _rowmajor(out, "out"), M, N, _ptr(bias), _ptr(rowbias),
                                              rowbias_div, _rowmajor(rowbias, "rowbias") if rowbias is not None else 0,
                                              _ptr(res1), _rowmajor(res1, "res1") if res1 is not None else 0,
                                              _ptr(res2), _rowmajor(res2, "res2") if res2 is not None else 0,
                                              _ptr(scales), int(act), _stream()), "svdx_splitk_epilogue_act")
        return out
    return tapgemm(a, b, out, M=M, N=N, K=K, taps=taps, bias=bias, rowbias=rowbias, rowbias_div=rowbias_div, res1=res1, res2=res2,
                   scales=scales, gn_sum=gn_sum, gn_rows=gn_rows, act=act, **kw)


def fill_rows(out: torch.Tensor, vec: torch.Tensor) -> torch.Tensor:
    """out[r, :] = bf16(vec) for every row of a bf16 [rows, N] view (any row stride): the split-K epilogue over its zeroed
    workspace with vec (fp32 [N]) as the bias (the CLIP class-token rows, one launch for the whole batch)"""
    rows, N = out.shape
    ws = _splitk_workspace(rows, N, out.device)
    check(load().svdx_splitk_epilogue_act(ws.data_ptr(), N, out.data_ptr(), _rowmajor(out, "out"), rows, N, vec.data_ptr(), None, 1, 0,
                                          None, 0, None, 0, None, ACT_NONE, _stream()), "svdx_splitk_epilogue_act")
    return out


CONV3x3_TAPS = tuple((kw - 1, kh - 1, 0) for kh in range(3) for kw in range(3))


# ----------------------------------------------------------------------------- attention
def _attn_desc(q, k, v, o, heads, S, nseq, inner, outer_stride, inner_stride, tok_stride, scale, lse):
    d = SvdxAttn()
    d.q, d.k, d.v, d.o = q.data_ptr(), k.data_ptr(), v.data_ptr(), o.data_ptr()
    d.ldq, d.ldk, d.ldv, d.ldo = _rowmajor(q, "q"), _rowmajor(k, "k"), _rowmajor(v, "v"), _rowmajor(o, "o")
    d.nseq, d.heads, d.S, d.inner = nseq, heads, S, inner
    d.outer_stride, d.inner_stride, d.tok_stride = outer_stride, inner_stride, tok_stride
    d.scale = scale
    d.lse = _ptr(lse)
    return d


def attention_fwd(q, k, v, o, *, heads, S, nseq, inner=1, outer_stride=None, inner_stride=0, tok_stride=1,
                  scale=0.125, lse=None):
    """q/k/v/o: [tokens, >=heads*64] bf16 (column slices allowed). Spatial: inner=1, outer_stride=S."""
    if outer_stride is None:
        outer_stride = S
    if _fam("attention", 4.0 * nseq * heads * S * S * 64):
        return o
    d = _attn_desc(q, k, v, o, heads, S, nseq, inner, outer_stride, inner_stride, tok_stride, scale, lse)
    check(load().svdx_attention_fwd(C.byref(d), _stream()), "svdx_attention_fwd")
    return o


def attention_vit(q, k, v, o, *, heads, S, nseq, scale=80 ** -0.5):
    """ViT self-attention, head_dim 80, forward only (svdx_attention_vit_fwd): q/k/v/o [nseq * S, >= heads*80] bf16 column
    slices (q, k, v usually of one fused [rows, 3C] q|k|v matrix); sequence s = rows [s*S, (s+1)*S)"""
    if _fam("attention", 4.0 * nseq * heads * S * S * 80):
        return o
    d = _attn_desc(q, k, v, o, heads, S, nseq, 1, S, 0, 1, scale, None)
    check(load().svdx_attention_vit_fwd(C.byref(d), _stream()), "svdx_attention_vit_fwd")
    return o


def attention_bwd(q, k, v, o, dout, dq, dk, dv, lse, delta, *, heads, S, nseq, inner=1, outer_stride=None,
                  inner_stride=0, tok_stride=1, scale=0.125):
    if outer_stride is None:
        outer_stride = S
    if _fam("attention", 10.0 * nseq * heads * S * S * 64):     # flash backward = 2.5 x forward (5 GEMMs of S^2 x 64)
        return
    d = _attn_desc(q, k, v, o, heads, S, nseq, inner, outer_stride, inner_stride, tok_stride, scale, lse)
    d.dout, d.lddo = dout.data_ptr(), _rowmajor(dout, "dout")
    d.dq, d.dk, d.dv = dq.data_ptr(), dk.data_ptr(), dv.data_ptr()
    d.lddq, d.lddk, d.lddv = _rowmajor(dq, "dq"), _rowmajor(dk, "dk"), _rowmajor(dv, "dv")
    d.delta = delta.data_ptr()
    check(load().svdx_attention_bwd(C.byref(d), _stream()), "svdx_attention_bwd")


# ----------------------------------------------------------------------------- norms
def groupnorm_stats(x, x2, outer, rows, eps, groups=32):
    C1 = x.shape[-1]
    C2 = x2.shape[-1] if x2 is not None else 0
    stats = torch.empty(2, outer * groups, device=x.device, dtype=torch.float32)   # adjacent: zeroed by ONE memset node
    mean, rstd = stats[0], stats[1]
    if _fam("groupnorm", 0.0, 2.0 * x.shape[0] * (C1 + C2)):
        return mean, rstd
    check(load().svdx_groupnorm_stats(x.data_ptr(), _rowmajor(x, "x"), C1, _ptr(x2), _rowmajor(x2, "x2") if x2 is not None else 0,
                                      C2, outer, rows, groups, eps, mean.data_ptr(), rstd.data_ptr(), _stream()), "svdx_groupnorm_stats")
    return mean, rstd


def groupnorm_apply(x, x2, outer, rows, mean, rstd, gamma, beta, silu, y, groups=32, ab=None):
    C1 = x.shape[-1]
    C2 = x2.shape[-1] if x2 is not None else 0
    if _fam("groupnorm", 0.0, 4.0 * x.shape[0] * (C1 + C2)):
        return y
    check(load().svdx_groupnorm_apply(x.data_ptr(), _rowmajor(x, "x"), C1, _ptr(x2), _rowmajor(x2, "x2") if x2 is not None else 0,
                                      C2, outer, rows, groups, mean.data_ptr(), rstd.data_ptr(), gamma.data_ptr(), beta.data_ptr(),
                                      int(silu), y.data_ptr(), _rowmajor(y, "y"), _ptr(ab), _stream()), "groupnorm_apply")
    return y


def groupnorm_apply_fused(x, x2, outer, rows, eps, csum1, csum2, gamma, beta, silu, y, groups=32, ab=None):
    """GroupNorm(+SiLU) from the per-channel sums of the producing epilogues; returns (mean, rstd) [outer*groups] for backward.
    ab: optional fp32 [outer, 2, C] that receives the per-channel scale / shift (for tapgemm's gnb_* backward sums)"""
    C1 = x.shape[-1]
    C2 = x2.shape[-1] if x2 is not None else 0
    stats = torch.empty(2, outer * groups, device=x.device, dtype=torch.float32)
    mean, rstd = stats[0], stats[1]
    if _fam("groupnorm", 0.0, 4.0 * x.shape[0] * (C1 + C2)):
        return mean, rstd
    check(load().svdx_groupnorm_apply_fused(x.data_ptr(), _rowmajor(x, "x"), C1, _ptr(x2), _rowmajor(x2, "x2") if x2 is not None else 0, C2,
                                            outer, rows, groups, eps, csum1.data_ptr(), csum1.shape[2],
                                            _ptr(csum2), csum2.shape[2] if csum2 is not None else 0, mean.data_ptr(), rstd.data_ptr(),
                                            gamma.data_ptr(), beta.data_ptr(), int(silu), y.data_ptr(), _rowmajor(y, "y"), _ptr(ab), _stream()),
          "svdx_groupnorm_apply_fused")
    return mean, rstd


def groupnorm_bwd(x, x2, dy, outer, rows, mean, rstd, gamma, beta, silu, dx, dx2, dgamma=None, dbeta=None, groups=32, ws=None, dres=None):
    """ws: optional pre-ZEROED float[2 * outer * groups] workspace (a slice of a zeroed arena: no memset node);
    dres: gradient already accumulated on x (bf16, same shape), added to dx in the same pass"""
    C1 = x.shape[-1]
    C2 = x2.shape[-1] if x2 is not None else 0
    ws_zero = ws is not None
    if ws is None:
        ws = torch.empty(outer * groups * 2, device=x.device, dtype=torch.float32)
    if _fam("groupnorm", 0.0, 6.0 * x.shape[0] * (C1 + C2)):       # minimal traffic: read x, dy once, write dx
        return
    check(load().svdx_groupnorm_bwd(x.data_ptr(), _rowmajor(x, "x"), C1, _ptr(x2), _rowmajor(x2, "x2") if x2 is not None else 0, C2,
                                    dy.data_ptr(), _rowmajor(dy, "dy"), outer, rows, groups, mean.data_ptr(), rstd.data_ptr(),
                                    gamma.data_ptr(), beta.data_ptr(), int(silu), dx.data_ptr(), _rowmajor(dx, "dx"),
                                    _ptr(dx2), _rowmajor(dx2, "dx2") if dx2 is not None else 0, _ptr(dgamma), _ptr(dbeta),
                                    ws.data_ptr(), int(ws_zero), _ptr(dres), _rowmajor(dres, "dres") if dres is not None else 0, _stream()),
          "svdx_groupnorm_bwd")


def groupnorm_bwd_fused(x, x2, dy, outer, rows, mean, rstd, gamma, beta, silu, csum, dx, dx2, dgamma=None, dbeta=None, groups=32, dres=None):
    """GroupNorm backward from the per-channel sums the dgrad epilogue accumulated (tapgemm gnb_sum): one launch, one pass"""
    C1 = x.shape[-1]
    C2 = x2.shape[-1] if x2 is not None else 0
    if _fam("groupnorm", 0.0, 6.0 * x.shape[0] * (C1 + C2)):
        return
    check(load().svdx_groupnorm_bwd_fused(x.data_ptr(), _rowmajor(x, "x"), C1, _ptr(x2), _rowmajor(x2, "x2") if x2 is not None else 0, C2,
                                          dy.data_ptr(), _rowmajor(dy, "dy"), outer, rows, groups, mean.data_ptr(), rstd.data_ptr(),
                                          gamma.data_ptr(), beta.data_ptr(), int(silu), csum.data_ptr(), dx.data_ptr(), _rowmajor(dx, "dx"),
                                          _ptr(dx2), _rowmajor(dx2, "dx2") if dx2 is not None else 0, _ptr(dgamma), _ptr(dbeta),
                                          _ptr(dres), _rowmajor(dres, "dres") if dres is not None else 0, _stream()),
          "svdx_groupnorm_bwd_fused")


def layernorm_fwd(x, gamma, beta, eps, y, addvec=None, add_div=1, xsum=None):
    rows, Cc = x.shape
    mean = torch.empty(rows, device=x.device, dtype=torch.float32)
    rstd = torch.empty_like(mean)
    if _fam("layernorm", 0.0, (6.0 if xsum is not None else 4.0) * rows * Cc):
        return mean, rstd
    check(load().svdx_layernorm_fwd(x.data_ptr(), _rowmajor(x, "x"), rows, Cc, gamma.data_ptr(), beta.data_ptr(), eps,
                                    y.data_ptr(), _rowmajor(y, "y"), mean.data_ptr(), rstd.data_ptr(), _ptr(addvec), add_div,
                                    _ptr(xsum), _rowmajor(xsum, "xsum") if xsum is not None else 0, _stream()), "layernorm_fwd")
    return mean, rstd


def layernorm_bwd(x, dy, gamma, mean, rstd, dx, dres=None, dgamma=None, dbeta=None):
    rows, Cc = x.shape
    if _fam("layernorm", 0.0, (8.0 if dres is not None else 6.0) * rows * Cc):
        return
    check(load().svdx_layernorm_bwd(x.data_ptr(), _rowmajor(x, "x"), dy.data_ptr(), _rowmajor(dy, "dy"), rows, Cc, gamma.data_ptr(),
                                    mean.data_ptr(), rstd.data_ptr(), dx.data_ptr(), _rowmajor(dx, "dx"), _ptr(dres),
                                    _rowmajor(dres, "dres") if dres is not None else 0, _ptr(dgamma), _ptr(dbeta), _stream()),
          "layernorm_bwd")


# ----------------------------------------------------------------------------- CLIP preprocessing
CLIP_SIZE = 224
CLIP_PATCH_K = 588       # 3 x 14 x 14 values of one patch
CLIP_PATCH_KP = 592      # padded to 16-byte rows


@functools.lru_cache(maxsize=None)
def clip_blur_taps(H: int, W: int):
    """(ky, kx, wy, wx, (sigma_y, sigma_x)) of the anti-aliasing blur applied before resampling an H x W image to 224 x 224
    (train_svd.py:140-162, 218-232): sigma = max((in / 224 - 1) / 2, 0.001) per axis, kernel size int(max(4 sigma, 3)) made
    odd, normalised Gaussian taps computed in float64"""
    sig = tuple(max((n / CLIP_SIZE - 1.0) / 2.0, 0.001) for n in (H, W))
    ks = []
    for s in sig:
        k = int(max(2.0 * 2 * s, 3))
        ks.append(k + 1 if k % 2 == 0 else k)
    taps = []
    for k, s in zip(ks, sig):
        g = [math.exp(-float(i - k // 2) ** 2 / (2.0 * s * s)) for i in range(k)]
        tot = math.fsum(g)
        taps.append(tuple(v / tot for v in g))
    return ks[0], ks[1], taps[0], taps[1], sig


def clip_pixels(x: torch.Tensor, out: torch.Tensor, *, resize: bool, mean=(0.0, 0.0, 0.0), std=(1.0, 1.0, 1.0)) -> torch.Tensor:
    """[B, 3, H, W] images -> bf16 patch matrix out [B*256, >= 592] (svdx_clip_pixels). resize=True: anti-aliased bicubic
    resize to 224 x 224, (x + 1) / 2, (x - mean) / std; resize=False: an already normalised 224 x 224 input, patchify only."""
    B, Cc, H, W = x.shape
    if Cc != 3 or not x.is_contiguous():
        raise ValueError("clip_pixels: x must be a contiguous [B, 3, H, W] tensor")
    if out.dtype != bf16 or out.dim() != 2 or out.shape[0] != B * 256 or out.shape[1] < CLIP_PATCH_KP:
        raise ValueError("clip_pixels: out must be a bf16 [B * 256, >= 592] matrix")
    d = SvdxClipPixels()
    d.x = x.data_ptr()
    d.dtype = dtype_code(x, "image")
    d.B, d.H, d.W = B, H, W
    d.resize = int(resize)
    if resize:
        ky, kx, wy, wx, _ = clip_blur_taps(H, W)
        if max(ky, kx) > _lib.SVDX_CLIP_MAX_TAPS:
            raise ValueError(f"clip_pixels: {H}x{W} needs a {ky}x{kx} blur; at most {_lib.SVDX_CLIP_MAX_TAPS} taps per axis are supported")
        d.ky, d.kx = ky, kx
        for i, v in enumerate(wy):
            d.wy[i] = v
        for i, v in enumerate(wx):
            d.wx[i] = v
    for i in range(3):
        d.mean[i], d.std[i] = float(mean[i]), float(std[i])
    d.out = out.data_ptr()
    d.ldo = _rowmajor(out, "out")
    check(load().svdx_clip_pixels(C.byref(d), _stream()), "svdx_clip_pixels")
    return out


# ----------------------------------------------------------------------------- elementwise / layout
def prep_weight(src, dst, mode, O, I, taps=1, i_pad=None):
    check(load().svdx_prep_weight(src.data_ptr(), dtype_code(src, "weight"), dst.data_ptr(), mode, O, I, taps,
                                  i_pad if i_pad is not None else I, _stream()), "prep_weight")
    return dst


def cast_f32_bf16(src, dst):
    if _fam("elementwise", 0.0, 6.0 * src.numel()):
        return dst
    check(load().svdx_cast_f32_bf16(src.data_ptr(), dst.data_ptr(), src.numel(), _stream()), "cast_f32_bf16")
    return dst


def cast_bf16_f32(src, dst):
    check(load().svdx_cast_bf16_f32(src.data_ptr(), dst.data_ptr(), src.numel(), _stream()), "cast_bf16_f32")
    return dst


def cast_to_f32(src, dst):
    """fp32 copy of a bf16 / fp16 vector (biases and norm affine vectors of a half-precision model)"""
    code = dtype_code(src, "vector")
    if code == 1:
        return cast_bf16_f32(src, dst)
    if code == 2:
        check(load().svdx_cast_f16_f32(src.data_ptr(), dst.data_ptr(), src.numel(), _stream()), "cast_f16_f32")
        return dst
    raise TypeError("cast_to_f32: source is already fp32")


def nchw_to_nhwc(src, dst, N, Cc, H, W, c_pad):
    check(load().svdx_nchw_to_nhwc(src.data_ptr(), dtype_code(src, "NCHW input"), dst.data_ptr(), N, Cc, H, W, c_pad, _stream()), "nchw_to_nhwc")
    return dst


def nhwc_to_nchw(src, dst, N, Cc, H, W):
    check(load().svdx_nhwc_to_nchw(src.data_ptr(), _rowmajor(src, "src"), dst.data_ptr(), dtype_code(dst, "NCHW output"), N, Cc, H, W, _stream()),
          "nhwc_to_nchw")
    return dst


def upsample2x(src, dst, N, H, W, Cc):
    check(load().svdx_upsample2x(src.data_ptr(), dst.data_ptr(), N, H, W, Cc, _stream()), "upsample2x")
    return dst


def upsample2x_bwd(dsrc, ddst, N, H, W, Cc):
    check(load().svdx_upsample2x_bwd(dsrc.data_ptr(), ddst.data_ptr(), N, H, W, Cc, _stream()), "upsample2x_bwd")
    return ddst


def space_to_planes(src, dst, N, H, W, Cc):
    check(load().svdx_space_to_planes(src.data_ptr(), dst.data_ptr(), N, H, W, Cc, _stream()), "space_to_planes")
    return dst


def planes_to_space(src, dst, N, H, W, Cc):
    check(load().svdx_planes_to_space(src.data_ptr(), dst.data_ptr(), N, H, W, Cc, _stream()), "planes_to_space")
    return dst


def concat_channels(a, b, dst):
    if _fam("elementwise", 0.0, 4.0 * dst.numel()):
        return dst
    check(load().svdx_concat_channels(a.data_ptr(), a.shape[-1], b.data_ptr(), b.shape[-1], dst.data_ptr(), a.numel() // a.shape[-1],
                                      _stream()), "concat_channels")
    return dst


def split_channels(src, a, b, accumulate_a=False):
    Ca = a.shape[-1]
    Cb = src.shape[-1] - Ca
    if _fam("elementwise", 0.0, 4.0 * src.numel()):
        return
    check(load().svdx_split_channels(src.data_ptr(), a.data_ptr(), Ca, _ptr(b), Cb, src.numel() // src.shape[-1], int(accumulate_a),
                                     _stream()), "split_channels")


def axpby(a, b, y, scales=None):
    if _fam("elementwise", 0.0, 6.0 * a.numel()):
        return y
    check(load().svdx_axpby_bf16(a.data_ptr(), b.data_ptr(), _ptr(scales), y.data_ptr(), a.numel(), _stream()), "axpby_bf16")
    return y


def silu_f32(x, y):
    check(load().svdx_silu_f32(x.data_ptr(), y.data_ptr(), x.numel(), _stream()), "silu_f32")
    return y


def colsum(x, out, accumulate=False):
    rows, cols = x.shape
    if _fam("elementwise", 0.0, 2.0 * rows * cols):
        return out
    check(load().svdx_colsum(x.data_ptr(), _rowmajor(x, "x"), rows, cols, out.data_ptr(), int(accumulate), _stream()), "colsum")
    return out


def geglu_bwd(pre, dout, dpre, bias_grad=None):
    """bias_grad: fp32 [2h] accumulator of the GEGLU projection's bias gradient (column sums of dpre, fused in the same pass)"""
    rows, h2 = pre.shape
    if _fam("elementwise", 0.0, 10.0 * rows * (h2 // 2)):
        return dpre
    check(load().svdx_geglu_bwd(pre.data_ptr(), _rowmajor(pre, "pre"), dout.data_ptr(), _rowmajor(dout, "dout"), dpre.data_ptr(),
                                _rowmajor(dpre, "dpre"), rows, h2 // 2, _ptr(bias_grad), _stream()), "geglu_bwd")
    return dpre


def gemv(a, w, out, *, M, N, K, bias=None, lda=None, ldw=None, scale=1.0, accumulate=False):
    """out[m, n] = scale * sum_k a[m, k] w[n, k] (+ bias[n]) (+ out[m, n]) for M <= 8 rows (conditioning vectors): weight-streaming GEMV"""
    if _fam("linear", 2.0 * M * N * K):
        return out
    check(load().svdx_gemv(a.data_ptr(), lda if lda is not None else _rowmajor(a, "a"), w.data_ptr(), ldw if ldw is not None else _rowmajor(w, "w"),
                           M, N, K, _ptr(bias), out.data_ptr(), _rowmajor(out, "out"), OUT_BF16 if out.dtype == bf16 else OUT_F32, float(scale),
                           int(accumulate), _stream()), "svdx_gemv")
    return out


def outer_accum(dy, x, g, scale=None):
    """g[o, k] += scale * sum_t dy[t, o] x[t, k] for T <= 8 token rows (weight gradient of a skinny product)"""
    T, O = dy.shape
    K = x.shape[1]
    if _fam("linear", 2.0 * T * O * K):
        return g
    check(load().svdx_outer_accum(dy.data_ptr(), _rowmajor(dy, "dy"), x.data_ptr(), _rowmajor(x, "x"), T, O, K, _ptr(scale), g.data_ptr(),
                                  _rowmajor(g, "g"), _stream()), "svdx_outer_accum")
    return g


def softmax_rows(x, y, scale=1.0):
    rows, cols = x.shape
    if _fam("elementwise", 0.0, 4.0 * rows * cols):
        return y
    check(load().svdx_softmax_rows(x.data_ptr(), _rowmajor(x, "x"), rows, cols, float(scale), y.data_ptr(), _rowmajor(y, "y"), _stream()),
          "svdx_softmax_rows")
    return y


def blend_scales(mix_factor, out3):  # out3: float[8]
    check(load().svdx_blend_scales(mix_factor.data_ptr(), out3.data_ptr(), _stream()), "blend_scales")
    return out3


def adamw(p, g, m, v, lr, beta1, beta2, eps, weight_decay, step, grad_scale=1.0, shadow=None):
    if _fam("adamw", 0.0, (30.0 if shadow is not None else 28.0) * p.numel()):
        return
    check(load().svdx_adamw(p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), p.numel(), lr, beta1, beta2, eps, weight_decay,
                            step, grad_scale, _ptr(shadow), _stream()), "adamw")


def adamw_p2p(p, m, v, peer_grads, peer_shadows, lo, state, grad_scale, tick=True):
    """reduce-scatter + AdamW + all-gather in one kernel over NVLink peer memory (svdx_adamw_p2p): p / m / v are this rank's
    slices, peer_grads / peer_shadows the FULL arenas of every rank (this rank's own included) as tensors mapped into this
    process (train.map_peer_buffers)"""
    world = len(peer_grads)
    n = p.numel()
    if _fam("adamw", 0.0, (4.0 * world + 28.0 + 2.0 * world) * n):
        return
    ga = (C.c_void_p * world)(*[t if isinstance(t, int) else t.data_ptr() for t in peer_grads])       # tensors or mapped addresses
    sa = (C.c_void_p * world)(*[t if isinstance(t, int) else t.data_ptr() for t in peer_shadows])
    check(load().svdx_adamw_p2p(p.data_ptr(), m.data_ptr(), v.data_ptr(), ga, sa, world, lo, n, state.data_ptr(), float(grad_scale),
                                int(tick), _stream()), "svdx_adamw_p2p")


def adamw_graph(p, g, m, v, state, grad_scale=1.0, shadow=None):
    """CUDA-graph-safe AdamW: lr / betas / eps / weight decay / step / bias corrections live in the device float[8] `state`"""
    if _fam("adamw", 0.0, (30.0 if shadow is not None else 28.0) * p.numel()):
        return
    check(load().svdx_adamw_graph(p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr(), p.numel(), state.data_ptr(), grad_scale,
                                  _ptr(shadow), _stream()), "svdx_adamw_graph")


def multi_transpose(src_base, jobs, tile_prefix, njobs, total_tiles):
    if _fam("elementwise", 0.0, 4.0 * 64 * 64 * total_tiles):
        return
    check(load().svdx_multi_transpose(src_base.data_ptr(), jobs.data_ptr(), tile_prefix.data_ptr(), njobs, total_tiles, _stream()),
          "svdx_multi_transpose")


def unprep_conv_grad(src, dst, O, I, taps, i_pad):
    check(load().svdx_unprep_conv_grad(src.data_ptr(), dst.data_ptr(), O, I, taps, i_pad, _stream()), "svdx_unprep_conv_grad")
    return dst


def dot_diff(dy, a, b, out):
    check(load().svdx_dot_diff(dy.data_ptr(), a.data_ptr(), b.data_ptr(), dy.numel(), out.data_ptr(), _stream()), "svdx_dot_diff")
    return out


def silu_bwd_f32(x, dy, dx):
    check(load().svdx_silu_bwd_f32(x.data_ptr(), dy.data_ptr(), dx.data_ptr(), x.numel(), _stream()), "svdx_silu_bwd_f32")
    return dx

/*
 * svd_xtend_b200 — C ABI of the B200-native SVD spatio-temporal UNet hot path.
 *
 * Every entry point takes raw device pointers, explicit shapes/strides and a CUDA stream
 * (passed as void* == cudaStream_t). Contract for ALL functions:
 *   - return 0 on success, <0 on error (see SVDX_E_*); never throw, never allocate or free
 *     device memory, never synchronise the device; re-entrant across streams;
 *   - bf16 = __nv_bfloat16 storage, fp32 accumulation everywhere.
 *
 * The reference (pixeli99/SVD_Xtend) is pure Python on top of diffusers; the operator each entry
 * replaces is therefore the ATen/cuDNN/cuBLAS call reached from the reference's module code.
 * The replaced interface is cited per function as  <reference file:line> -> <diffusers op [D]>.
 * "[D]" = code that lives in the un-vendored diffusers dependency (SURVEY.md Appendix B).
 */
#ifndef SVD_XTEND_B200_H_
#define SVD_XTEND_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SVDX_OK 0
#define SVDX_E_BADARG (-1)     /* unsupported shape / alignment / null pointer */
#define SVDX_E_CUDA (-2)       /* CUDA runtime / driver error on launch */
#define SVDX_E_NODRIVER (-3)   /* cuTensorMapEncodeTiled entry point unavailable */

#define SVDX_MAX_TAPS 27

/* A-operand addressing modes of svdx_tapgemm */
#define SVDX_A_ROWS 0    /* A is [groups][rows_per_group][K] (a plain matrix when groups==1);
                            tap t reads rows shifted by tap_d0[t] inside the group, rows outside
                            the group read as zero (this is the (3,1,1) temporal conv / a linear) */
#define SVDX_A_CONV2D 1  /* A is [nimg][H][W][K] channels-last; tap t reads pixel (h+tap_d1[t],
                            w+tap_d0[t]) of image n+tap_d2[t]; out-of-image reads are zero
                            (3x3 conv padding=1, and the parity-plane form of the stride-2 conv) */

#define SVDX_OUT_BF16 0
#define SVDX_OUT_F32 1
#define SVDX_OUT_F32_ATOMIC 2  /* out += result (fp32 red.add), used by split-K weight gradients */

/*
 * svdx_tapgemm — the one tensor-core contraction of the path (tcgen05.mma, TMEM accumulators,
 * TMA-fed 128B-swizzled shared memory, warp-specialised persistent CTAs):
 *
 *     acc[m, n] = sum_{t < num_taps} sum_{k < K}  A_t[m, k] * B[n, t*K + k]
 *     v         = acc + bias[n] + rowbias[m / rowbias_div, n]
 *     v         = geglu ? v[:, :N/2] * gelu_erf(v[:, N/2:]) : v
 *     out[m, n] = scales[0] * v + scales[1] * res1[m, n] + scales[2] * res2[m, n]
 *
 * Replaces, with the epilogue fused:
 *   F.linear      — Attention.to_q/to_k/to_v/to_out, FeedForward proj/out, proj_in/proj_out,
 *                   time_emb_proj, TimestepEmbedding  [D]; reached from
 *                   src/unet_spatio_temporal_condition.py:138-144,170-233
 *   F.conv2d 3x3  — ResnetBlock2D.conv1/conv2, Downsample2D, Upsample2D.conv [D], conv_in/conv_out
 *                   (src/unet_spatio_temporal_condition.py:128-133,241-246)
 *   F.conv2d 1x1  — ResnetBlock2D.conv_shortcut [D]
 *   F.conv3d (3,1,1) — TemporalResnetBlock.conv1/conv2 [D]
 *   GEGLU, AlphaBlender, residual adds [D] (epilogue)
 * and their data/weight gradients (dgrad = same contraction on transposed weights; wgrad =
 * a_major_mn = b_major_mn = 1 with SVDX_OUT_F32_ATOMIC).
 */
typedef struct SvdxTapGemm {
  /* A operand (bf16) */
  const void* a;
  int64_t lda;          /* elements between consecutive rows/pixels */
  int32_t a_mode;       /* SVDX_A_ROWS / SVDX_A_CONV2D */
  int32_t a_major_mn;   /* 0: A[m][k] k contiguous. 1 (ROWS, groups==1 only): memory is [k][m], m contiguous */
  int32_t rows_per_group, groups;      /* ROWS   */
  int32_t W, H, nimg;                  /* CONV2D: 128 % W == 0, or W % 128 == 0 (wide images: a tile is 128 pixels of one row) */
  int32_t num_taps;
  int32_t tap_d0[SVDX_MAX_TAPS];
  int32_t tap_d1[SVDX_MAX_TAPS];
  int32_t tap_d2[SVDX_MAX_TAPS];
  /* B operand (bf16): [N][num_taps*K] (k contiguous), or if b_major_mn: memory [K][N], n contiguous */
  const void* b;
  int64_t ldb;
  int32_t b_major_mn;
  int32_t b_mode;       /* weight-gradient forms (a_major_mn = b_major_mn = 1): 0 plain [K][N];
                           1: B is a channels-last image tensor [nimg][H][W][N], contraction row p (an output
                              pixel) reads pixel shifted by (tap_d0[0], tap_d1[0]) of image +tap_d2[0], zero outside
                              (dW of a 3x3 conv tap); K = images*H*W output pixels;
                           2: B is [groups][rows_per_group][N], contraction row reads row + tap_d0[0] of its
                              group, zero outside (dW of a (3,1,1) temporal conv tap) */
  /* problem */
  int32_t M, N, K;      /* M output rows, N = B rows (before GEGLU halving), K = contraction per tap */
  int32_t block_n;      /* multiple of 32, <= 256 (multiple of 64 when b_major_mn); 320 = the CTA-pair kernel's 256 x 320 tile
                           (two N = 160 MMAs per k-step on one A stage): M >= 512, N % 320 == 0, bf16 TMA-store epilogues only */
  int32_t split_k;      /* >= 1; > 1 requires SVDX_OUT_F32_ATOMIC */
  /* epilogue */
  void* out;
  int64_t ldo;
  int32_t out_dtype;
  int32_t geglu;        /* out has N/2 columns */
  const float* bias;    /* [N] or NULL */
  const float* rowbias; /* [ceil(M/rowbias_div)][ldrb] or NULL */
  int32_t rowbias_div;
  int64_t ldrb;
  const void* res1;     /* bf16 [M][ldr1] or NULL */
  int64_t ldr1;
  const void* res2;
  int64_t ldr2;
  const float* scales;  /* device float[3] {acc, res1, res2} or NULL (= 1,1,1) */
  void* pre;            /* geglu: bf16 [M][ldpre] pre-activation (value | gate) saved for backward, or NULL */
  int64_t ldpre;
  /* GroupNorm statistics of the OUTPUT, fused into the epilogue ("GroupNorm fused into the conv epilogue"): when gn_sum is
   * not NULL the epilogue also accumulates, per statistics slab s = m / gn_rows and output channel n, the sum and the sum
   * of squares of the bf16 values it stores:  gn_sum[(2*s + 0) * gn_ld + n] += out[m][n],  gn_sum[(2*s + 1) * gn_ld + n] +=
   * out[m][n]^2  (fp32 red.add; column sums of each staged 32x32 chunk, warp-reduced). gn_rows = rows per slab (H*W per
   * frame for the spatial GroupNorms, T*H*W per clip for the temporal ones); the buffer must be zero on entry. The consumer
   * (svdx_groupnorm_apply_fused) folds channels into groups, so a later channel concatenation needs no extra pass.
   * Requires a bf16 output written through the TMA-store epilogues (N % 32 == 0, 16-byte aligned rows), no split-K, no GEGLU. */
  float* gn_sum;
  int64_t gn_ld;        /* floats per (slab, moment) row, >= N */
  int32_t gn_rows;
  /* GroupNorm BACKWARD statistics fused into the epilogue (pass 1 of F.group_norm's backward): set on the GEMM / conv that
   * WRITES dy = dL/d(GroupNorm output) — the data gradient of the conv that consumed the normalised tensor. gnb_x (channels
   * [0, gnb_c1)) and gnb_x2 (the rest; NULL = single source) are the GroupNorm's bf16 INPUT, gnb_ab[(2*s + 0) * N + n] /
   * [(2*s + 1) * N + n] the forward scale / shift of channel n in statistics slab s = m / gnb_rows (written by
   * svdx_groupnorm_apply*, y = act(x * scale + shift); only read when gnb_silu). The epilogue accumulates
   *   gnb_sum[(2*s + 0) * N + n] += e,  gnb_sum[(2*s + 1) * N + n] += e * x[m][n],   e = dy[m][n] * act'(x * scale + shift)
   * on the bf16 values it stores (buffer zero on entry); svdx_groupnorm_bwd_fused turns them into dx / dgamma / dbeta with ONE
   * pass over x and dy. Requires the plain bf16 TMA-store epilogue (no residual / scales / GEGLU / split-K / gn_sum), N even. */
  const void* gnb_x;
  int64_t gnb_ldx;
  const void* gnb_x2;
  int64_t gnb_ldx2;
  int32_t gnb_c1;
  const float* gnb_ab;
  float* gnb_sum;
  int32_t gnb_rows;
  int32_t gnb_silu;
  /* activation of the accumulator (SVDX_ACT_*), applied before the residual / scale step:
   *   v = act(acc + bias + rowbias),  out = scales[0] * v + scales[1] * res1 + scales[2] * res2.
   * SVDX_ACT_GELU replaces the F.gelu of CLIPMLP (transformers CLIPVisionModelWithProjection, loaded at train_svd.py:646 and run
   * at :875) on fc1's output. Requires a bf16 output, no GEGLU, no gn_sum / gnb_* statistics; with split_k > 1 the activation
   * belongs to the second pass (svdx_splitk_epilogue_act). Zero (the default of a zero-initialised descriptor) = none. */
  int32_t act;
} SvdxTapGemm;

#define SVDX_ACT_NONE 0
#define SVDX_ACT_GELU 1   /* gelu(x) = x * Phi(x), the erf form (hidden_act "gelu") */

int svdx_tapgemm(const SvdxTapGemm* desc, void* stream);

/* Second half of a split-K svdx_tapgemm (fp32 partial sums accumulated with SVDX_OUT_F32_ATOMIC into ws): applies the
 * same epilogue  out = scales[0]*(ws + bias + rowbias[m / rowbias_div]) + scales[1]*res1 + scales[2]*res2  -> bf16.
 * Used for the 5x8 / 10x16 latent levels where M gives too few output tiles to fill 148 SMs.
 * The workspace is CONSUMED: every element read is reset to zero, so a caller can keep one zeroed workspace per shape
 * and never memset it again. */
int svdx_splitk_epilogue(float* ws, int64_t ldw, void* out, int64_t ldo, int64_t rows, int32_t cols, const float* bias,
                         const float* rowbias, int32_t rowbias_div, int64_t ldrb, const void* res1, int64_t ldr1,
                         const void* res2, int64_t ldr2, const float* scales, void* stream);
/* the same second pass with an activation (SVDX_ACT_*) applied before the residual step:
 *   out = scales[0] * act(ws + bias + rowbias) + scales[1] * res1 + scales[2] * res2.
 * Used for CLIPMLP.fc1 + F.gelu (train_svd.py:875 -> transformers CLIPMLP) at B = 1, where the 257-row GEMM has 3 row tiles. */
int svdx_splitk_epilogue_act(float* ws, int64_t ldw, void* out, int64_t ldo, int64_t rows, int32_t cols, const float* bias,
                             const float* rowbias, int32_t rowbias_div, int64_t ldrb, const void* res1, int64_t ldr1,
                             const void* res2, int64_t ldr2, const float* scales, int32_t act, void* stream);

/* number of SMs the persistent kernels size their grids to (queried once) */
int svdx_num_sms(void);
/* enable peer access from the current device to peer_device (needed before svdx_adamw_p2p dereferences arenas that live on,
 * or were IPC-mapped from, that GPU); idempotent; fails when the GPUs have no P2P path */
int svdx_enable_peer_access(int32_t peer_device);
/* CUDA IPC of a device buffer between the processes of one node (one process per GPU). export: the 64-byte handle of the
 * allocation that contains ptr + ptr's byte offset inside it. import (call it with the CONSUMING GPU current): maps the
 * allocation into this process for that GPU (peer access enabled lazily) and returns the address corresponding to ptr. An
 * allocation can be imported once per process; the mapping lives until the process exits. */
int svdx_ipc_export(const void* ptr, void* handle64_out, int64_t* offset_out);
int svdx_ipc_import(const void* handle64, int64_t offset, void** ptr_out);
/* sizeof(SvdxTapGemm) (which==0) / sizeof(SvdxAttn) (which==1) / sizeof(SvdxClipPixels) (which==2): lets bindings verify
 * their struct layout */
int svdx_struct_size(int which);
/* human-readable last error of this thread */
const char* svdx_last_error(void);

/* ------------------------------------------------------------------ normalisation
 * GroupNorm(32)+SiLU over channels-last activations, replaces F.group_norm + F.silu of
 * ResnetBlock2D.norm1/norm2, TemporalResnetBlock.norm1/norm2 (stats over T*H*W),
 * TransformerSpatioTemporalModel.norm [D], conv_norm_out (src/unet_spatio_temporal_condition.py:238-239,480-481).
 * x is [ngroups_outer][rows][C] bf16 where one statistics group spans `rows` rows x (C/32) channels.
 * A second source x2 (C2 channels) is concatenated along channels (the up-block torch.cat).
 */
int svdx_groupnorm_stats(const void* x, int64_t ldx, int32_t C1, const void* x2, int64_t ldx2, int32_t C2,
                         int32_t outer, int32_t rows, int32_t num_groups, float eps,
                         float* mean, float* rstd, void* stream);
int svdx_groupnorm_apply(const void* x, int64_t ldx, int32_t C1, const void* x2, int64_t ldx2, int32_t C2,
                         int32_t outer, int32_t rows, int32_t num_groups,
                         const float* mean, const float* rstd, const float* gamma, const float* beta,
                         int32_t fuse_silu, void* y, int64_t ldy, float* ab_out, void* stream);
/* ab_out (optional, both apply forms): fp32 [outer][2][C], receives the per-channel scale / shift of every slab
 * (y = act(x * scale + shift)) — the gnb_ab table of the GroupNorm-backward sums fused into svdx_tapgemm's epilogue.
 * gamma / beta must be 16-byte aligned.
 *
 * GroupNorm(+SiLU) apply from per-CHANNEL sums produced by the svdx_tapgemm epilogues (gn_sum above): csum1 / csum2 are the
 * [outer][2][ld] fp32 sum / sum-of-squares arrays of the two channel-concatenated sources (csum2 NULL when C2 == 0). Every
 * CTA first folds the channels of its slab into the 32 group statistics (shared memory), the CTA with blockIdx.x == 0 of
 * each slab also writes mean / rstd [outer][groups] for the backward. Replaces stats + finalize + apply by ONE launch. */
int svdx_groupnorm_apply_fused(const void* x, int64_t ldx, int32_t C1, const void* x2, int64_t ldx2, int32_t C2,
                               int32_t outer, int32_t rows, int32_t num_groups, float eps,
                               const float* csum1, int64_t ldc1, const float* csum2, int64_t ldc2,
                               float* mean, float* rstd, const float* gamma, const float* beta,
                               int32_t fuse_silu, void* y, int64_t ldy, float* ab_out, void* stream);
/* backward: dx (and optional dgamma/dbeta accumulation, fp32 atomic). workspace: float[2 * outer * groups]; it must be
 * ZERO on entry when workspace_is_zero != 0 (a slice of a pre-zeroed arena: no memset node), else it is cleared here.
 * dres (optional, bf16 [outer*rows][lddres], single-source form only): a gradient already accumulated on x through its
 * residual use; dx = GroupNorm backward + dres in the same pass (replaces a separate bf16 add over the activation). */
int svdx_groupnorm_bwd(const void* x, int64_t ldx, int32_t C1, const void* x2, int64_t ldx2, int32_t C2,
                       const void* dy, int64_t lddy,
                       int32_t outer, int32_t rows, int32_t num_groups,
                       const float* mean, const float* rstd, const float* gamma, const float* beta,
                       int32_t fuse_silu, void* dx, int64_t lddx, void* dx2, int64_t lddx2,
                       float* dgamma, float* dbeta, float* workspace, int32_t workspace_is_zero,
                       const void* dres, int64_t lddres, void* stream);
/* backward when pass 1 already ran inside the epilogue that produced dy (svdx_tapgemm gnb_sum): csum = that [outer][2][C]
 * buffer (sum e, sum e*x per slab and channel). One launch, one pass over x and dy: every CTA folds the channel sums into the
 * group sums, dgamma / dbeta (optional, accumulated) come straight from the channel sums. Other arguments as svdx_groupnorm_bwd. */
int svdx_groupnorm_bwd_fused(const void* x, int64_t ldx, int32_t C1, const void* x2, int64_t ldx2, int32_t C2,
                             const void* dy, int64_t lddy, int32_t outer, int32_t rows, int32_t num_groups,
                             const float* mean, const float* rstd, const float* gamma, const float* beta,
                             int32_t fuse_silu, const float* csum, void* dx, int64_t lddx, void* dx2, int64_t lddx2,
                             float* dgamma, float* dbeta, const void* dres, int64_t lddres, void* stream);

/* LayerNorm over the last dim (C <= 2560, C % 8 == 0), replaces F.layer_norm of
 * BasicTransformerBlock.norm1-3 / TemporalBasicTransformerBlock.norm_in,norm1-3 [D].
 * addvec (optional, [ceil(rows/add_div)][C] fp32): row r gets addvec[r / add_div] added before normalisation and
 * the bf16 sum is written to xsum (the "hidden_states + emb" of TransformerSpatioTemporalModel [D]). */
int svdx_layernorm_fwd(const void* x, int64_t ldx, int32_t rows, int32_t C, const float* gamma, const float* beta,
                       float eps, void* y, int64_t ldy, float* mean, float* rstd,
                       const float* addvec, int32_t add_div, void* xsum, int64_t ldxs, void* stream);
int svdx_layernorm_bwd(const void* x, int64_t ldx, const void* dy, int64_t lddy, int32_t rows, int32_t C,
                       const float* gamma, const float* mean, const float* rstd,
                       void* dx, int64_t lddx, const void* dres, int64_t lddres,
                       float* dgamma, float* dbeta, void* stream);

/* ------------------------------------------------------------------ attention
 * Scaled-dot-product attention, head_dim 64, no mask, replaces
 * AttnProcessor2_0 -> F.scaled_dot_product_attention [D].
 * q/k/v/o are column slices of token-major [tokens][ld] bf16 matrices; head h uses columns
 * [h*64, h*64+64). A sequence s (0 <= s < nseq) has its i-th token at row  seq_base(s) + i*tok_stride
 * with seq_base(s) = (s / inner) * outer_stride + (s % inner) * inner_stride:
 *   spatial  (per frame over H*W):  inner = 1,  outer_stride = HW, tok_stride = 1
 *   temporal (per pixel over T):    inner = HW, outer_stride = T*HW, inner_stride = 1, tok_stride = HW
 * lse [nseq][heads][S] fp32 (natural-log sum-exp of the scaled scores) is saved for backward. */
typedef struct SvdxAttn {
  const void* q; const void* k; const void* v; void* o;
  int64_t ldq, ldk, ldv, ldo;
  int32_t nseq, heads, S;
  int32_t inner;
  int64_t outer_stride, inner_stride, tok_stride;
  float scale;
  float* lse;
  /* backward only */
  const void* dout; int64_t lddo;
  void* dq; void* dk; void* dv; int64_t lddq, lddk, lddv;
  float* delta;     /* workspace [nseq][heads][S] */
} SvdxAttn;
int svdx_attention_fwd(const SvdxAttn* d, void* stream);
int svdx_attention_bwd(const SvdxAttn* d, void* stream);
/* ViT self-attention of the CLIP image encoder, forward only: head_dim 80 (head h = columns [h*80, h*80+80), 160-byte
 * offsets), no mask, 1 <= S <= 512 tokens per sequence (257 for ViT-H/14), sequences are contiguous blocks of rows
 * (inner = 1, tok_stride = 1, outer_stride >= S; nseq = images). q / k / v may be column slices of one fused [tokens][3C]
 * q|k|v matrix; o is written at the same head columns only. lse / backward fields are ignored. One launch per layer, no S x S
 * matrix in memory. Replaces CLIPAttention's softmax(q k^T * scale) v (transformers, reached from train_svd.py:875). */
int svdx_attention_vit_fwd(const SvdxAttn* d, void* stream);

/* ------------------------------------------------------------------ CLIP image preprocessing
 * svdx_clip_pixels: [B][3][H][W] images (NCHW contiguous, dtype code 0/1/2) -> the bf16 patch matrix of the ViT patch
 * embedding, [B * 256][ldo] with row b * 256 + py * 16 + px holding the 3 * 14 * 14 = 588 values of patch (py, px) in
 * (c, ky, kx) order (= patch_embedding.weight.view(C, 588)), columns 588 .. 591 zero (ldo >= 592, ldo % 8 == 0).
 *   resize = 1 (encode_image, train_svd.py:857-876): separable Gaussian blur (taps wy[ky] / wx[kx], odd sizes <= 31, reflect
 *              padding of (k - 1) / 2, as _gaussian_blur2d / _filter2d, train_svd.py:193-248), then bicubic align_corners=True
 *              resampling to 224 x 224 (A = -0.75, source index dst * (in - 1) / 223, neighbours clamped: F.interpolate of
 *              _resize_with_antialiasing, train_svd.py:140-167), then (x + 1) / 2 and (x - mean[c]) / std[c]
 *              (CLIPImageProcessor(do_normalize=True, ...), train_svd.py:864-871). The host computes the taps per (H, W).
 *              The arithmetic is float64 end to end (taps, source coordinates, cubic weights, sums, normalisation), so the
 *              bf16 result is the correctly rounded value of the exact resize up to ties: in float32 the source coordinate
 *              dst * (in - 1) / 223 alone carries ~1e-4 of error at the far edge, and cancellation around the mean leaves
 *              values near zero with few correct bits. 14 <= H, 14 <= W <= 6144.
 *   resize = 0 (CLIPVisionModelWithProjection(pixel_values)): H = W = 224, already normalised: patchify only.
 * Replaces ~10 torch ops and the image processor's host round trip with one launch. */
#define SVDX_CLIP_MAX_TAPS 31
typedef struct SvdxClipPixels {
  const void* x;
  int32_t dtype;        /* 0 fp32, 1 bf16, 2 fp16 */
  int32_t B, H, W;
  int32_t resize;
  int32_t ky, kx;       /* blur taps along H / W (resize = 1) */
  double wy[SVDX_CLIP_MAX_TAPS];
  double wx[SVDX_CLIP_MAX_TAPS];
  double mean[3], std[3];
  void* out;
  int64_t ldo;
} SvdxClipPixels;
int svdx_clip_pixels(const SvdxClipPixels* d, void* stream);

/* ------------------------------------------------------------------ elementwise / layout */
/* weights -> bf16, optionally re-laid-out. src_bf16 is the SOURCE DTYPE CODE used by every entry of this section:
 * 0 = fp32, 1 = bf16, 2 = fp16 (train_svd_lora.py:669 moves the frozen UNet to fp16 / bf16 `weight_dtype`).
 *   mode 0: plain copy           dst[n][k]           = src[n][k]
 *   mode 1: transpose            dst[k][n]           = src[n][k]            (dgrad operand of a linear)
 *   mode 2: conv OIHW -> O(HW)I  dst[o][t][i(pad)]   = src[o][i][t]         (fwd operand; taps = kh*kw or kt)
 *   mode 3: conv OIHW -> I(HW)O  dst[i][t][o]        = src[o][i][t]         (dgrad operand; the caller negates tap offsets)
 * i_pad >= I pads the input-channel axis with zeros (conv_in: 8 -> 64). */
int svdx_prep_weight(const void* src, int32_t src_bf16, void* dst, int32_t mode,
                     int32_t O, int32_t I, int32_t taps, int32_t i_pad, void* stream);
/* adjoint of svdx_prep_weight mode 2: dst[o][i][t] += src[o][t][i] (fp32; src row = taps*i_pad, dst = OIHW gradient) */
int svdx_unprep_conv_grad(const float* src, float* dst, int32_t O, int32_t I, int32_t taps, int32_t i_pad, void* stream);
/* sum over all elements of dy * (a - b) (bf16 inputs) accumulated into out[0] (fp32): AlphaBlender mix_factor gradient */
int svdx_dot_diff(const void* dy, const void* a, const void* b, int64_t n, float* out, void* stream);
/* y = dy * silu'(x) on fp32 vectors (time-embedding MLP backward) */
int svdx_silu_bwd_f32(const float* x, const float* dy, float* dx, int64_t n, void* stream);
int svdx_cast_f32_bf16(const float* src, void* dst, int64_t n, void* stream);
int svdx_cast_bf16_f32(const void* src, float* dst, int64_t n, void* stream);
int svdx_cast_f16_f32(const void* src, float* dst, int64_t n, void* stream);
/* NCHW (dtype code 0/1/2) -> [N][H][W][c_pad] bf16 (zero padded channels) and back (to an NCHW tensor of dtype code dst_bf16) */
int svdx_nchw_to_nhwc(const void* src, int32_t src_bf16, void* dst, int32_t N, int32_t C, int32_t H, int32_t W,
                      int32_t c_pad, void* stream);
int svdx_nhwc_to_nchw(const void* src, int64_t lds, void* dst, int32_t dst_bf16, int32_t N, int32_t C, int32_t H,
                      int32_t W, void* stream);
/* nearest 2x upsample, channels-last (F.interpolate of Upsample2D [D]) and its adjoint (2x2 sum) */
int svdx_upsample2x(const void* src, void* dst, int32_t N, int32_t H, int32_t W, int32_t C, void* stream);
int svdx_upsample2x_bwd(const void* dsrc, void* ddst, int32_t N, int32_t H, int32_t W, int32_t C, void* stream);
/* parity planes for the stride-2 conv: dst[(p*2+q)*N + n][H/2][W/2][C] = src[n][2h+p][2w+q][C], and adjoint */
int svdx_space_to_planes(const void* src, void* dst, int32_t N, int32_t H, int32_t W, int32_t C, void* stream);
int svdx_planes_to_space(const void* src, void* dst, int32_t N, int32_t H, int32_t W, int32_t C, void* stream);
/* channel concat / split of channels-last tensors (torch.cat(dim=1) of the up blocks) */
int svdx_concat_channels(const void* a, int32_t Ca, const void* b, int32_t Cb, void* dst, int64_t rows, void* stream);
int svdx_split_channels(const void* src, void* a, int32_t Ca, void* b, int32_t Cb, int64_t rows, int32_t accumulate_a,
                        void* stream);
/* y = a + b (bf16), y = silu(x) for fp32 vectors, column sums (bias gradients) */
int svdx_add_bf16(const void* a, const void* b, void* y, int64_t n, void* stream);
int svdx_axpby_bf16(const void* a, const void* b, const float* scales, void* y, int64_t n, void* stream);
int svdx_silu_f32(const float* x, float* y, int64_t n, void* stream);
int svdx_colsum(const void* x, int64_t ldx, int64_t rows, int32_t cols, float* out, int32_t accumulate, void* stream);
/* GEGLU backward: dpre[m][:h] = dout*gelu(gate); dpre[m][h:] = dout*value*gelu'(gate). bias_grad (optional, fp32 [2h], accumulated):
 * += column sums of the dpre values written — the bias gradient of the GEGLU projection, fused into the same pass */
int svdx_geglu_bwd(const void* pre, int64_t ldpre, const void* dout, int64_t lddo, void* dpre, int64_t lddpre,
                   int64_t rows, int32_t h, float* bias_grad, void* stream);
/* y[r][:] = softmax(scale * x[r][:]) over bf16 rows (fp32 arithmetic, in place allowed). Used by the VAE encoder's mid-block
 * attention (1 head of dim 512, [D] AutoencoderKLTemporalDecoder.encoder.mid_block.attentions.0): scores = Q K^T and P V go through
 * svdx_tapgemm, the row softmax through this kernel. */
int svdx_softmax_rows(const void* x, int64_t ldx, int64_t rows, int32_t cols, float scale, void* y, int64_t ldy, void* stream);
/* Skinny products of the per-clip conditioning vectors ([B, C] rows: TimestepEmbedding MLPs, every resnet's time_emb_proj, the
 * 1-key image cross-attention to_out(to_v(e)) [D], their LoRA side paths and their data gradients):
 *   out[m][n] = scale * sum_k a[m][k] * w[n][k] + bias[n]  (+ out[m][n] when accumulate != 0),
 * M <= 8 rows, bf16 operands, fp32 accumulation, bf16 (SVDX_OUT_BF16) or fp32 (SVDX_OUT_F32) output. A weight-streaming GEMV
 * (one warp per output column): the 128-row tensor-core tiles of svdx_tapgemm would be > 99 % padding here. */
int svdx_gemv(const void* a, int64_t lda, const void* w, int64_t ldw, int32_t M, int32_t N, int32_t K, const float* bias,
              void* out, int64_t ldo, int32_t out_dtype, float scale, int32_t accumulate, void* stream);
/* ...and their weight gradients: g[o][k] += scale[0] * sum_{t < T} dy[t][o] * x[t][k], T <= 8 (scale NULL = 1) */
int svdx_outer_accum(const void* dy, int64_t lddy, const void* x, int64_t ldx, int32_t T, int32_t O, int32_t K,
                     const float* scale, float* g, int64_t ldg, void* stream);
/* AlphaBlender epilogue scale triples from mix_factor, a = sigmoid(mix_factor); writes float[16]:
 *   out[0..3]   = {1-a, a, 1-a, 0}      transformer blend  out = a*x_spatial + (1-a)*(acc + residual)
 *   out[4..7]   = {1-a, 1, 0, a*(1-a)}  resnet blend       out = x_spatial + (1-a)*acc
 *   out[8..11]  = {1-a, 0, 0, 0}        accumulator-only triple (gradient GEMMs of a blended forward)
 *   out[12..15] = {a, 0, 1-a, 0}        {s, 0} pairs for svdx_axpby_bf16 (gradients of the residual operands) */
int svdx_blend_scales(const float* mix_factor, float* out16, void* stream);
/* fused multi-tensor AdamW on a flat fp32 buffer (torch.optim.AdamW of train_svd.py:767-773); when shadow_bf16 is given
 * the updated parameters are also written as bf16 at the same flat offsets (the forward GEMM operands) */
int svdx_adamw(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2,
               float eps, float weight_decay, int32_t step, float grad_scale, void* shadow_bf16, void* stream);
/* the same update with every step-varying scalar in DEVICE memory, so that it can be captured in a CUDA graph and replayed:
 * state = float[8] {lr, beta1, beta2, eps, weight_decay, step, 1-beta1^step, 1-beta2^step}. The call first advances
 * step and the bias corrections on the device (a 1-thread kernel), then updates; the host changes the learning rate by
 * writing state[0] (lr scheduler of train_svd.py:790-796). Two launches. */
int svdx_adamw_graph(float* p, const float* g, float* m, float* v, int64_t n, float* state, float grad_scale,
                     void* shadow_bf16, void* stream);
/* Data-parallel optimizer step over NVLink peer memory (one process per GPU, every rank's gradient and bf16 operand arenas
 * mapped into every process with CUDA IPC): reduce-scatter + AdamW + all-gather as ONE kernel. This rank owns [lo, lo + n):
 * it loads that slice of grads[r] (r = 0 .. world-1, the FULL arenas, peer-mapped), sums in rank order, applies AdamW with
 * grad_scale (= 1 / world) to its local p / m / v slices (length n) and stores the bf16 value to shadows[r][lo + i] of every
 * rank. The caller provides the cross-rank ordering: all gradients final before the launch, no rank reads its shadow or
 * clears its gradients until every rank's launch has completed. tick != 0 also advances the device step count / bias
 * corrections in state[5..7] (svdx_adamw_graph's state layout). Replaces DistributedDataParallel's all-reduce +
 * torch.optim.AdamW of train_svd.py:767-773,815-824,1044-1049 at N > 1. */
int svdx_adamw_p2p(float* p, float* m, float* v, const void* const* grads, void* const* shadows, int32_t world,
                   int64_t lo, int64_t n, float* state, float grad_scale, int32_t tick, void* stream);

/* many bf16 transposes dst[i][o] = src_base[src_off + o*I + i] in one launch (dgrad operands of all trainable linears).
 * jobs: device array of {int64 src_off; void* dst; int32 O; int32 I}; tile_prefix[j] = first 32x32 tile of job j. */
int svdx_multi_transpose(const void* src_base, const void* jobs, const int32_t* tile_prefix, int32_t njobs, int32_t total_tiles,
                         void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SVD_XTEND_B200_H_ */

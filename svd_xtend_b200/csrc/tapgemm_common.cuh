// Shared pieces of the tcgen05 tapgemm kernels (1-CTA in tapgemm.cu, 2-CTA pairs in tapgemm2.cu):
// kernel parameter block, tile geometry and the fused epilogue of one accumulator tile.
#pragma once
#include "common.cuh"
#include "../../include/svd_xtend_b200.h"
#include "host_util.h"

// default of the SVDX_2CTA switch (env SVDX_2CTA=0/1 overrides): use the CTA-pair kernel where eligible
#ifndef SVDX_2CTA_DEFAULT
#define SVDX_2CTA_DEFAULT 1
#endif

namespace svdx {

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;
constexpr int STAGES = 4;
constexpr int A_STAGE_BYTES = BLOCK_M * BLOCK_K * 2;  // 16 KB
constexpr int B_STAGE_BYTES = 256 * BLOCK_K * 2;      // 32 KB
constexpr int ACC_STAGES = 2;
constexpr int TMEM_COLS = 512;
constexpr int NUM_EPI_WARPS = 8;   // two warps per TMEM lane quarter, each takes every other 32-column chunk
constexpr int NUM_THREADS = 64 + 32 * NUM_EPI_WARPS;
constexpr int EPI_STAGE_BYTES = 4096;  // per epilogue warp: 2 x (32 rows x 64 B) bf16 halves or 1 x (32 rows x 128 B) fp32
constexpr int SMEM_BYTES = 1024 + STAGES * (A_STAGE_BYTES + B_STAGE_BYTES) + NUM_EPI_WARPS * EPI_STAGE_BYTES + 256;

struct __align__(64) TapGemmKParams {
  CUtensorMap tma;
  CUtensorMap tmb;
  CUtensorMap tma_bh[4];  // CONV2D: boxes of 2, 4, 8, 16 image rows (tma itself = 1 row)
  int max_bh_log2;
  int a_mode, a_mn, b_mn, b_mode, kb_per_group;
  int rows_per_group, groups, tiles_per_group;
  int W, H, nimg;
  int wtiles;          // CONV2D with W > 128 (W % 128 == 0): a tile = 128 consecutive pixels of ONE image row, wtiles = W / 128 (else 0)
  int num_taps;
  int tap_d0[SVDX_MAX_TAPS], tap_d1[SVDX_MAX_TAPS], tap_d2[SVDX_MAX_TAPS];
  int M, N, K;
  int block_n, m_tiles, n_tiles, split_k, kb_total, kb_per_split, kb_per_tap;
  int pair_m_tiles, tiles_per_group_pairs;   // CTA-pair kernel: 256-row tiles (never straddling a group)
  // epilogue
  void* out;
  long long ldo;
  int out_dtype, geglu;
  const float* bias;
  const float* rowbias;
  int rowbias_div;
  long long ldrb;
  const bf16* res1;
  long long ldr1;
  const bf16* res2;
  long long ldr2;
  const float* scales;
  bf16* pre;
  long long ldpre;
  CUtensorMap tmo;     // output (bf16: 32x32 box, 64B swizzle; fp32: 32x32 box, 128B swizzle), dims {n_out, rows, groups}
  CUtensorMap tmpre;   // GEGLU pre-activation [M, N]
  float* gn_sum;       // fused GroupNorm statistics of the output (per slab m / gn_rows, per channel): [slab][2][gn_ld]
  long long gn_ld;
  int gn_rows;
  // GroupNorm BACKWARD statistics fused into the epilogue of the GEMM / conv that writes dy = dL/d(GroupNorm output)
  const bf16* gnb_x;   // the GroupNorm's INPUT (channels [0, gnb_c1)), and gnb_x2 the concatenated second source
  long long gnb_ldx;
  const bf16* gnb_x2;
  long long gnb_ldx2;
  int gnb_c1;
  const float* gnb_ab; // [slab][2][N]: forward scale / shift per channel (y = act(x * scale + shift))
  float* gnb_sum;      // [slab][2][N], zero on entry: sum(e), sum(e * x), e = dy * act'(x * scale + shift)
  int gnb_rows, gnb_silu;
  int act;             // SVDX_ACT_*: activation of acc + bias + rowbias, before residuals / scales
  int tma_store;       // epilogue stores through shared memory + TMA (tmo / tmpre valid)
  int epi_mode;        // EPI_GENERIC / EPI_FAST / EPI_GEGLU / EPI_RES: which kernel instantiation runs
  int probe;   // dev switch SVDX_EPI_PROBE: 1 = epilogue without global stores, 2 = no epilogue work at all
};


// output row of epilogue thread r (0..127) of m-tile mt, and whether it exists
SVDX_DEVINL void tile_row(const TapGemmKParams& p, int mt, int r, long long& m, bool& row_ok) {
  if (p.a_mode == SVDX_A_ROWS && !p.a_mn) {
    const int g = mt / p.tiles_per_group;
    const int t = mt - g * p.tiles_per_group;
    const int rin = t * BLOCK_M + r;
    row_ok = rin < p.rows_per_group;
    m = (long long)g * p.rows_per_group + rin;
  } else {
    m = (long long)mt * BLOCK_M + r;
    row_ok = m < p.M;
  }
}

// ---- conv A tiles: the 128 pixels of a tile are R = 128 / W consecutive image rows, fetched as a few multi-row TMA
// boxes (image borders and tile/image straddling decide the split). The split depends on the tile only, so it is
// computed once per tile with lane l of the producer warp keeping box l; per k-block every lane that owns a box
// issues its TMA. (The per-k-block scalar decomposition cost ~1.5-3 k cycles and made the producer thread the
// bottleneck of every 3x3 convolution: profiles/r1_conv_probe.txt.)
struct ConvBox {
  int lg, hh, n;
  uint32_t dst_off;
  bool nvalid, active;
};
SVDX_DEVINL void conv_tile_boxes(const TapGemmKParams& p, int t, int lane, ConvBox& mine) {
  const int R = BLOCK_M / p.W;
  int rowid = t * R, left = R, idx = 0;
  uint32_t off = 0;
  mine.active = false; mine.lg = 0; mine.hh = 0; mine.n = 0; mine.dst_off = 0; mine.nvalid = false;
  while (left > 0) {
    const int n = rowid / p.H;
    const int h = rowid - n * p.H;
    int run = min(left, p.H - h);
    int hh = h;
    while (run > 0) {
      const int lg = min(p.max_bh_log2, 31 - __clz(run));
      const int bh = 1 << lg;
      if (idx == lane) { mine.lg = lg; mine.hh = hh; mine.n = n; mine.nvalid = n < p.nimg; mine.dst_off = off; mine.active = true; }
      off += bh * p.W * 128;
      hh += bh; run -= bh; left -= bh; rowid += bh; ++idx;
    }
  }
}

// ---- staged stores: a warp writes its 32-row x 32-column chunk into shared memory (one row per lane, swizzled so
// that the 16-byte writes are conflict-free) and one lane hands it to the TMA unit. The global writes become full
// 64/128-byte row segments issued asynchronously, instead of 32 scattered 16-byte sectors per store instruction
// (measured: the scattered stores made every K<=640 GEMM epilogue-bound, profiles/r1_epilogue_probe.txt).
// Rows past the end of the group / matrix and columns past n_out are clipped by the tensor map.
struct EpiStage {
  uint32_t base;   // this warp's 4 KB staging region (1024-aligned)
  uint32_t off;    // bf16: alternates between the two 2 KB halves
  int row0, grp;   // tensor-map coordinates of this warp's first row
};

SVDX_DEVINL void stage_store_bf16(const CUtensorMap* tm, EpiStage& st, int lane, const float (&f)[32], int col) {
  if (lane == 0) bulk_wait_read<1>();   // the half written two stores ago has been read out
  __syncwarp();
  const uint32_t buf = st.base + st.off;
  const uint32_t row = buf + lane * 64;
  const int sw = (lane >> 1) & 3;       // CU_TENSOR_MAP_SWIZZLE_64B: 16-byte chunk index ^= address bits [7:8]
#pragma unroll
  for (int j = 0; j < 4; ++j)
    st_shared_v4(row + ((j ^ sw) << 4), pack_bf16x2(f[8 * j], f[8 * j + 1]), pack_bf16x2(f[8 * j + 2], f[8 * j + 3]),
                 pack_bf16x2(f[8 * j + 4], f[8 * j + 5]), pack_bf16x2(f[8 * j + 6], f[8 * j + 7]));
  fence_proxy_async_smem();
  __syncwarp();
  if (lane == 0) { tma_store_3d(tm, buf, col, st.row0, st.grp); bulk_commit(); }
  st.off ^= 2048;
}

SVDX_DEVINL void stage_store_f32(const CUtensorMap* tm, EpiStage& st, int lane, const float (&f)[32], int col, bool reduce) {
  if (lane == 0) bulk_wait_read<0>();
  __syncwarp();
  const uint32_t row = st.base + lane * 128;
  const int sw = lane & 7;              // CU_TENSOR_MAP_SWIZZLE_128B
#pragma unroll
  for (int j = 0; j < 8; ++j)
    st_shared_v4(row + ((j ^ sw) << 4), __float_as_uint(f[4 * j]), __float_as_uint(f[4 * j + 1]), __float_as_uint(f[4 * j + 2]),
                 __float_as_uint(f[4 * j + 3]));
  fence_proxy_async_smem();
  __syncwarp();
  if (lane == 0) {
    if (reduce) tma_reduce_add_3d(tm, st.base, col, st.row0, st.grp);
    else tma_store_3d(tm, st.base, col, st.row0, st.grp);
    bulk_commit();
  }
}

// ---- GroupNorm statistics of the output, fused into the epilogue: column sums (and sums of squares) of one staged
// 32-row x 32-column bf16 chunk, i.e. of exactly the values the TMA store writes. Lane l takes the column pair l % 16 and
// the rows of parity l / 16 (two 64-byte rows per wavefront: conflict-free with the 64B swizzle), the two halves are
// combined with one shuffle and lanes 0..15 issue two red.global.add.v2.f32. Rows are walked slab by slab (a slab = gn_rows
// consecutive rows = one frame or one clip), so tiles that straddle frames (5x8 latents) stay correct.
// m0 = global row index of the chunk's row 0, valid_rows = how many of its 32 rows exist.
SVDX_DEVINL void gn_chunk_sums(const TapGemmKParams& p, uint32_t buf, int lane, int col0, int n_out_total, long long m0, int valid_rows) {
  const int pr = lane & 15, h = lane >> 4;
  const uint32_t in_chunk = (uint32_t)(pr & 3) * 4u;
  const int jch = pr >> 2;
  long long slab = m0 / p.gn_rows;
  int left = p.gn_rows - (int)(m0 - slab * p.gn_rows);
  int r = 0;
  while (r < valid_rows) {                                     // warp-uniform trip count
    const int seg_end = min(valid_rows, r + left);
    float s0 = 0.f, s1 = 0.f, q0 = 0.f, q1 = 0.f;
    for (int rr = r + ((h ^ r) & 1); rr < seg_end; rr += 2) {
      uint32_t w;
      asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w) : "r"(buf + rr * 64 + ((uint32_t)(jch ^ ((rr >> 1) & 3)) << 4) + in_chunk));
      const float2 v = unpack_bf16x2(w);
      s0 += v.x; s1 += v.y;
      q0 = fmaf(v.x, v.x, q0); q1 = fmaf(v.y, v.y, q1);
    }
    s0 += __shfl_xor_sync(0xffffffffu, s0, 16); s1 += __shfl_xor_sync(0xffffffffu, s1, 16);
    q0 += __shfl_xor_sync(0xffffffffu, q0, 16); q1 += __shfl_xor_sync(0xffffffffu, q1, 16);
    const int col = col0 + 2 * pr;
    if (h == 0 && col < n_out_total) {
      float* d = p.gn_sum + (2 * slab) * p.gn_ld + col;
      asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(d), "f"(s0), "f"(s1) : "memory");
      asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(d + p.gn_ld), "f"(q0), "f"(q1) : "memory");
    }
    r = seg_end; ++slab; left = p.gn_rows;
  }
}

// ---- specialised epilogues (kernel template parameter EPI): the hot shapes have short K, so the per-chunk instruction
// count of the epilogue decides their speed (profiles/r1_epilogue_probe.txt). EPI_FAST / EPI_GEGLU assume a bf16 output
// written through TMA, whole 32-column chunks (n_out % 32 == 0) and 16-byte aligned bias rows; everything else takes
// the generic epilogue_tile below.
constexpr int EPI_GENERIC = 0, EPI_FAST = 1, EPI_GEGLU = 2, EPI_RES = 3;
// + fused GroupNorm statistics of the output (separate instantiations: the plain ones keep their register budget)
constexpr int EPI_FAST_GN = 4, EPI_RES_GN = 5;
// + fused GroupNorm BACKWARD sums (the output is the gradient of a GroupNorm's output)
constexpr int EPI_FAST_GNB = 6;

SVDX_DEVINL void add_vec32(float (&f)[32], const float* __restrict__ src) {
  const float4* bp = reinterpret_cast<const float4*>(src);
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const float4 b4 = __ldg(bp + k);
    f[4 * k] += b4.x; f[4 * k + 1] += b4.y; f[4 * k + 2] += b4.z; f[4 * k + 3] += b4.w;
  }
}
SVDX_DEVINL void axpy_bf16x32(float (&f)[32], float s, const uint4 (&r)[4]) {
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const float2 a = unpack_bf16x2(r[k].x), b = unpack_bf16x2(r[k].y), c = unpack_bf16x2(r[k].z), d = unpack_bf16x2(r[k].w);
    f[8 * k] += s * a.x; f[8 * k + 1] += s * a.y; f[8 * k + 2] += s * b.x; f[8 * k + 3] += s * b.y;
    f[8 * k + 4] += s * c.x; f[8 * k + 5] += s * c.y; f[8 * k + 6] += s * d.x; f[8 * k + 7] += s * d.y;
  }
}
// one lane's 32 values -> its 64-byte row of a staging half (64B-swizzled)
SVDX_DEVINL void stage_row_bf16(uint32_t row, int sw, const float (&f)[32]) {
#pragma unroll
  for (int j = 0; j < 4; ++j)
    st_shared_v4(row + ((j ^ sw) << 4), pack_bf16x2(f[8 * j], f[8 * j + 1]), pack_bf16x2(f[8 * j + 2], f[8 * j + 3]),
                 pack_bf16x2(f[8 * j + 4], f[8 * j + 5]), pack_bf16x2(f[8 * j + 6], f[8 * j + 7]));
}

// activation of one 32-column chunk (p.act, warp-uniform)
SVDX_DEVINL void act32(float (&f)[32], int act) {
  if (act == SVDX_ACT_GELU) {
#pragma unroll
    for (int i = 0; i < 32; ++i) f[i] = gelu_erf_f(f[i]);
  }
}

// Epilogue operands that are read per chunk (the residual of EPI_RES, the GroupNorm input of EPI_FAST_GNB) are usually not in L2
// any more; a warp has ONE chunk's loads in flight, so the fetch was latency-bound (+12 us on a 15 us K = 320 residual GEMM,
// +20 us on a conv dgrad with the backward sums). Each epilogue warp therefore requests its 32 rows x bn columns of the tile
// into L2 BEFORE it waits for the accumulator: the lines arrive during the main loop. Lane = row; the two warps of a lane
// quarter take alternate 128-byte lines.
SVDX_DEVINL void prefetch_rows_l2(const bf16* base, long long ld, long long m0, int valid_rows, int col0, int ncols, int lane, int half) {
  if (!base || lane >= valid_rows) return;
  const char* row = reinterpret_cast<const char*>(base + (m0 + lane) * ld + col0);
  const int bytes = ncols * 2;
  for (int b = half * 128; b < bytes; b += 256) asm volatile("prefetch.global.L2 [%0];" ::"l"(row + b));
}
SVDX_DEVINL void prefetch_epilogue_operands(const TapGemmKParams& p, int epi, long long m0, int valid_rows, int n0, int bn_out, int n_out_total,
                                            int lane, int half) {
  const int ncols = min(bn_out, n_out_total - n0);
  if (ncols <= 0) return;
  if (epi == EPI_RES || epi == EPI_RES_GN) {
    prefetch_rows_l2(p.res1, p.ldr1, m0, valid_rows, n0, ncols, lane, half);
    prefetch_rows_l2(p.res2, p.ldr2, m0, valid_rows, n0, ncols, lane, half);
  } else if (epi == EPI_FAST_GNB) {
    if (n0 < p.gnb_c1) prefetch_rows_l2(p.gnb_x, p.gnb_ldx, m0, valid_rows, n0, min(ncols, p.gnb_c1 - n0), lane, half);
    if (n0 + ncols > p.gnb_c1) {
      const int c0 = max(n0, p.gnb_c1);
      prefetch_rows_l2(p.gnb_x2, p.gnb_ldx2, m0, valid_rows, c0 - p.gnb_c1, n0 + ncols - c0, lane, half);
    }
  }
}

// plain epilogue (bias / row-bias only): two 32-column chunks per round (both staging halves), one proxy fence and one
// bulk group per round.
template <bool GN>
SVDX_DEVINL void epilogue_fast(const TapGemmKParams& p, uint32_t t_base, long long m, bool row_ok, int n0, int half, int c_lo, int c_hi,
                               int n_out_total, uint32_t sbase, int row0, int grp, int lane, long long m0, int valid_rows) {
  const float* bias = p.bias;
  const float* rb = (p.rowbias && row_ok) ? p.rowbias + (m / p.rowbias_div) * p.ldrb : nullptr;
  const uint32_t rowX = sbase + lane * 64, rowY = rowX + 2048;
  const int sw = (lane >> 1) & 3;
#pragma unroll 1
  for (int c = c_lo + half * 32; c < c_hi; c += 128) {           // accumulator columns [c_lo, c_hi) of the tile
    const int colA = n0 + c;
    if (colA >= n_out_total) break;
    const int colB = colA + 64;
    const bool hasB = (c + 64 < c_hi) && (colB < n_out_total);     // warp-uniform
    uint32_t va[32], vb[32];
    tmem_ld32(t_base + c, va);
    if (hasB) tmem_ld32(t_base + c + 64, vb);
    tc_wait_ld();
    float fa[32], fb[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) { fa[i] = __uint_as_float(va[i]); fb[i] = __uint_as_float(vb[i]); }
    if (bias) { add_vec32(fa, bias + colA); if (hasB) add_vec32(fb, bias + colB); }
    if (rb) { add_vec32(fa, rb + colA); if (hasB) add_vec32(fb, rb + colB); }
    if (p.act) { act32(fa, p.act); if (hasB) act32(fb, p.act); }
    if (lane == 0) bulk_wait_read<0>();   // the previous round's stores have drained both halves
    __syncwarp();
    stage_row_bf16(rowX, sw, fa);
    if (hasB) stage_row_bf16(rowY, sw, fb);
    fence_proxy_async_smem();
    __syncwarp();
    if (lane == 0) {
      tma_store_3d(&p.tmo, sbase, colA, row0, grp);
      if (hasB) tma_store_3d(&p.tmo, sbase + 2048, colB, row0, grp);
      bulk_commit();
    }
    if constexpr (GN) {
      gn_chunk_sums(p, sbase, lane, colA, n_out_total, m0, valid_rows);
      if (hasB) gn_chunk_sums(p, sbase + 2048, lane, colB, n_out_total, m0, valid_rows);
    }
  }
}

// ---- GroupNorm backward, pass 1, fused into the epilogue that WRITES dy (the dgrad conv / GEMM whose input was the
// GroupNorm(+SiLU) output): per (slab, channel) S = sum_rows e and SX = sum_rows e * x with e = dy * act'(x * scale + shift),
// from the staged bf16 dy chunk (exactly the values stored) and the matching 32 x 32 chunk of the GroupNorm input x staged
// beside it. The consumer (svdx_groupnorm_bwd_fused) folds channels into groups: s1 = sum_c gamma_c S_c,
// s2 = rstd * (sum_c gamma_c SX_c - mean * s1); dgamma_c = rstd * (SX_c - mean * S_c), dbeta_c = S_c. Same lane layout as
// gn_chunk_sums (lane = column pair x row parity), slabs walked segment by segment.
SVDX_DEVINL void gnb_chunk_sums(const TapGemmKParams& p, uint32_t buf_dy, uint32_t buf_x, int lane, int col0, int n_out_total, long long m0,
                                int valid_rows) {
  const int pr = lane & 15, h = lane >> 4;
  const uint32_t in_chunk = (uint32_t)(pr & 3) * 4u;
  const int jch = pr >> 2;
  long long slab = m0 / p.gnb_rows;
  int left = p.gnb_rows - (int)(m0 - slab * p.gnb_rows);
  const int col = col0 + 2 * pr;
  const bool col_ok = col < n_out_total;
  int r = 0;
  while (r < valid_rows) {                                     // warp-uniform trip count
    const int seg_end = min(valid_rows, r + left);
    float2 A = make_float2(0.f, 0.f), B = make_float2(0.f, 0.f);
    if (col_ok && p.gnb_silu) {
      A = *reinterpret_cast<const float2*>(p.gnb_ab + (2 * slab) * p.N + col);
      B = *reinterpret_cast<const float2*>(p.gnb_ab + (2 * slab + 1) * p.N + col);
    }
    float s0 = 0.f, s1 = 0.f, x0 = 0.f, x1 = 0.f;
    if (r == 0 && seg_end == 32) {
      // the common case (a whole 32-row chunk inside one slab): rows h, h + 2, ... in two unrolled batches of 8 so that the
      // sigmoid chains (ex2 -> rcp) of different rows overlap; the rolled loop below ran one dependent chain at a time
#pragma unroll
      for (int b = 0; b < 2; ++b) {
        uint32_t wd[8], wx[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int rr = h + 2 * (8 * b + i);
          const uint32_t off = rr * 64 + ((uint32_t)(jch ^ ((rr >> 1) & 3)) << 4) + in_chunk;
          asm volatile("ld.shared.u32 %0, [%1];" : "=r"(wd[i]) : "r"(buf_dy + off));
          asm volatile("ld.shared.u32 %0, [%1];" : "=r"(wx[i]) : "r"(buf_x + off));
        }
        float e0[8], e1[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float2 d = unpack_bf16x2(wd[i]), xv = unpack_bf16x2(wx[i]);
          e0[i] = d.x; e1[i] = d.y;
          if (p.gnb_silu) {
            e0[i] *= silu_grad_f(fmaf(xv.x, A.x, B.x));
            e1[i] *= silu_grad_f(fmaf(xv.y, A.y, B.y));
          }
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float2 xv = unpack_bf16x2(wx[i]);
          s0 += e0[i]; s1 += e1[i];
          x0 = fmaf(e0[i], xv.x, x0); x1 = fmaf(e1[i], xv.y, x1);
        }
      }
    } else {
      for (int rr = r + ((h ^ r) & 1); rr < seg_end; rr += 2) {
        const uint32_t off = rr * 64 + ((uint32_t)(jch ^ ((rr >> 1) & 3)) << 4) + in_chunk;
        uint32_t wd, wx;
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(wd) : "r"(buf_dy + off));
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(wx) : "r"(buf_x + off));
        const float2 d = unpack_bf16x2(wd), xv = unpack_bf16x2(wx);
        float e0 = d.x, e1 = d.y;
        if (p.gnb_silu) {
          e0 *= silu_grad_f(fmaf(xv.x, A.x, B.x));
          e1 *= silu_grad_f(fmaf(xv.y, A.y, B.y));
        }
        s0 += e0; s1 += e1;
        x0 = fmaf(e0, xv.x, x0); x1 = fmaf(e1, xv.y, x1);
      }
    }
    s0 += __shfl_xor_sync(0xffffffffu, s0, 16); s1 += __shfl_xor_sync(0xffffffffu, s1, 16);
    x0 += __shfl_xor_sync(0xffffffffu, x0, 16); x1 += __shfl_xor_sync(0xffffffffu, x1, 16);
    if (h == 0 && col_ok) {
      float* d = p.gnb_sum + (2 * slab) * p.N + col;
      asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(d), "f"(s0), "f"(s1) : "memory");
      asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(d + p.N), "f"(x0), "f"(x1) : "memory");
    }
    r = seg_end; ++slab; left = p.gnb_rows;
  }
}

// plain epilogue + gnb_chunk_sums: one chunk per round, staging half X = the dy chunk (TMA-store source), half Y = the x chunk
SVDX_DEVINL void epilogue_fast_gnb(const TapGemmKParams& p, uint32_t t_base, long long m, bool row_ok, int n0, int half, int c_lo, int c_hi,
                                   int n_out_total, uint32_t sbase, int row0, int grp, int lane, long long m0, int valid_rows) {
  const float* bias = p.bias;
  const float* rb = (p.rowbias && row_ok) ? p.rowbias + (m / p.rowbias_div) * p.ldrb : nullptr;
  const uint32_t rowX = sbase + lane * 64;
  const int sw = (lane >> 1) & 3;
  const int prow = lane >> 2, ppc = lane & 3;
#pragma unroll 1
  for (int c = c_lo + half * 32; c < c_hi; c += 64) {
    const int col0 = n0 + c;
    if (col0 >= n_out_total) break;
    // the matching chunk of the GroupNorm input, fetched coalesced (8 rows x 64 B per instruction) before the TMEM wait
    const bool src1 = col0 < p.gnb_c1;
    const long long xld = src1 ? p.gnb_ldx : p.gnb_ldx2;
    const bf16* xs = (src1 ? p.gnb_x + col0 : p.gnb_x2 + (col0 - p.gnb_c1)) + m0 * xld + ppc * 8;
    uint4 xa[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int rr = prow + 8 * j;
      xa[j] = (rr < valid_rows) ? *reinterpret_cast<const uint4*>(xs + (long long)rr * xld) : make_uint4(0u, 0u, 0u, 0u);
    }
    uint32_t v[32];
    tmem_ld32(t_base + c, v);
    tc_wait_ld();
    float f[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) f[i] = __uint_as_float(v[i]);
    if (bias) add_vec32(f, bias + col0);
    if (rb) add_vec32(f, rb + col0);
    if (lane == 0) bulk_wait_read<0>();   // the previous round's store has drained half X
    __syncwarp();
    stage_row_bf16(rowX, sw, f);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int rr = prow + 8 * j;
      st_shared_v4(sbase + 2048 + rr * 64 + ((ppc ^ ((rr >> 1) & 3)) << 4), xa[j].x, xa[j].y, xa[j].z, xa[j].w);
    }
    fence_proxy_async_smem();
    __syncwarp();
    if (lane == 0) { tma_store_3d(&p.tmo, sbase, col0, row0, grp); bulk_commit(); }
    gnb_chunk_sums(p, sbase, sbase + 2048, lane, col0, n_out_total, m0, valid_rows);
    __syncwarp();                          // all lanes are done with half Y before the next round overwrites it
  }
}

// residual / AlphaBlender epilogue: out = s_acc*(acc + bias + rowbias) + s_r1*res1 + s_r2*res2; one chunk per round,
// alternating staging halves; the residual rows are requested before the TMEM wait.
template <bool GN>
SVDX_DEVINL void epilogue_res(const TapGemmKParams& p, uint32_t t_base, long long m, bool row_ok, int n0, int half, int c_lo, int c_hi,
                              int n_out_total, float s_acc, float s_r1, float s_r2, uint32_t sbase, uint32_t& off, int row0, int grp, int lane,
                              long long m0, int valid_rows) {
  const float* bias = p.bias;
  const float* rb = (p.rowbias && row_ok) ? p.rowbias + (m / p.rowbias_div) * p.ldrb : nullptr;
  // res1 (every residual add of the network) is fetched COALESCED: lane l loads the 16-byte piece l % 4 of rows l / 4 + 8 j
  // (8 rows x 64 B = 8 cache lines per instruction instead of one line per lane: the row-per-lane form cost 32 L1 tag
  // cycles per load and made the K = 320 / 640 residual GEMMs LSU-bound), the pieces are transposed through the staging half
  // that is about to receive this chunk's output, and every lane reads back its own row. res2 (AlphaBlender only) stays direct.
  const bf16* r1 = p.res1 ? p.res1 + m0 * p.ldr1 : nullptr;
  const bf16* r2 = (p.res2 && row_ok) ? p.res2 + m * p.ldr2 : nullptr;
  const bool scaled = p.scales != nullptr;
  const uint32_t row = sbase + lane * 64;
  const int sw = (lane >> 1) & 3;
  const int prow = lane >> 2, ppc = lane & 3;
  // `off` (which staging half comes next) lives in the caller across tiles: bulk_wait_read<1> only guarantees that the
  // half written TWO stores ago has been read out
#pragma unroll 1
  for (int c = c_lo + half * 32; c < c_hi; c += 64) {
    const int col0 = n0 + c;
    if (col0 >= n_out_total) break;
    uint4 a1[4], a2[4];
    if (r1) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int rr = prow + 8 * j;
        a1[j] = (rr < valid_rows) ? *reinterpret_cast<const uint4*>(r1 + (long long)rr * p.ldr1 + col0 + ppc * 8) : make_uint4(0u, 0u, 0u, 0u);
      }
    }
    if (r2) {
      const uint4* q = reinterpret_cast<const uint4*>(r2 + col0);
#pragma unroll
      for (int k = 0; k < 4; ++k) a2[k] = q[k];
    }
    uint32_t v[32];
    tmem_ld32(t_base + c, v);
    tc_wait_ld();
    float f[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) f[i] = __uint_as_float(v[i]);
    if (bias) add_vec32(f, bias + col0);
    if (rb) add_vec32(f, rb + col0);
    if (p.act) act32(f, p.act);
    if (scaled) {
#pragma unroll
      for (int i = 0; i < 32; ++i) f[i] *= s_acc;
    }
    if (lane == 0) bulk_wait_read<1>();
    __syncwarp();
    if (r1) {
      // transpose the coalesced pieces through the (now free) staging half: same 64B swizzle as the output rows
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int rr = prow + 8 * j;
        st_shared_v4(sbase + off + rr * 64 + ((ppc ^ ((rr >> 1) & 3)) << 4), a1[j].x, a1[j].y, a1[j].z, a1[j].w);
      }
      __syncwarp();
#pragma unroll
      for (int k = 0; k < 4; ++k)
        asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(a1[k].x), "=r"(a1[k].y), "=r"(a1[k].z), "=r"(a1[k].w) : "r"(row + off + ((k ^ sw) << 4)));
      axpy_bf16x32(f, s_r1, a1);
    }
    if (r2) axpy_bf16x32(f, s_r2, a2);
    stage_row_bf16(row + off, sw, f);
    fence_proxy_async_smem();
    __syncwarp();
    if (lane == 0) { tma_store_3d(&p.tmo, sbase + off, col0, row0, grp); bulk_commit(); }
    if constexpr (GN) gn_chunk_sums(p, sbase + off, lane, col0, n_out_total, m0, valid_rows);
    off ^= 2048;
  }
}

// GEGLU epilogue: value | gate column halves of the accumulator; optionally saves the bf16 pre-activation for backward.
SVDX_DEVINL void epilogue_geglu(const TapGemmKParams& p, uint32_t t_base, int n0, int half, int bn_out, uint32_t sbase, int row0,
                                int grp, int lane) {
  const float* bias = p.bias;
  const bool save_pre = p.pre != nullptr;
  const int nh = p.N / 2;
  const uint32_t rowX = sbase + lane * 64, rowY = rowX + 2048;
  const int sw = (lane >> 1) & 3;
  uint32_t off = 0;
#pragma unroll 1
  for (int c = half * 32; c < bn_out; c += 64) {
    const int col0 = n0 + c;
    uint32_t v[32], gte[32];
    tmem_ld32(t_base + c, v);
    tmem_ld32(t_base + bn_out + c, gte);
    tc_wait_ld();
    float f[32], g[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) { f[i] = __uint_as_float(v[i]); g[i] = __uint_as_float(gte[i]); }
    if (bias) { add_vec32(f, bias + col0); add_vec32(g, bias + nh + col0); }
    if (save_pre) {
      if (lane == 0) bulk_wait_read<0>();
      __syncwarp();
      stage_row_bf16(rowX, sw, f);
      stage_row_bf16(rowY, sw, g);
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        tma_store_3d(&p.tmpre, sbase, col0, row0, grp);
        tma_store_3d(&p.tmpre, sbase + 2048, nh + col0, row0, grp);
        bulk_commit();
      }
    }
    // the reference applies GEGLU on the bf16-rounded projection (autocast F.linear output)
#pragma unroll
    for (int i = 0; i < 32; ++i) {
      const float fv = __bfloat162float(__float2bfloat16(f[i]));
      const float gv = __bfloat162float(__float2bfloat16(g[i]));
      f[i] = fv * gelu_erf_f(gv);
    }
    if (save_pre) {
      if (lane == 0) bulk_wait_read<0>();
    } else {
      if (lane == 0) bulk_wait_read<1>();
    }
    __syncwarp();
    stage_row_bf16(save_pre ? rowX : rowX + off, sw, f);
    fence_proxy_async_smem();
    __syncwarp();
    if (lane == 0) { tma_store_3d(&p.tmo, save_pre ? sbase : sbase + off, col0, row0, grp); bulk_commit(); }
    off ^= 2048;
  }
}

// Epilogue of one accumulator tile for one thread (= one TMEM lane = one output row): this warp takes the 32-column
// chunks half, half+2, ...; bias / row-bias / GEGLU / residuals / scales, then staged TMA stores (or direct 16-byte
// stores when the output cannot be described by a tensor map).
SVDX_DEVINL void epilogue_tile(const TapGemmKParams& p, uint32_t t_base, long long m, bool row_ok, int n0, int half, int bn_out,
                               int n_out_total, float s_acc, float s_r1, float s_r2, EpiStage& st, int lane) {
      if (p.probe == 2) return;
      const float* rb = (p.rowbias && row_ok) ? p.rowbias + (m / p.rowbias_div) * p.ldrb : nullptr;
      for (int c = half * 32; c < bn_out; c += 64) {
        uint32_t v[32];
        uint32_t gte[32];
        const int col0 = n0 + c;
        if (col0 >= n_out_total) break;   // warp-uniform
        const bool full_chunk = (col0 + 32 <= n_out_total);
        // issue the global reads of this chunk before waiting on TMEM so their latency overlaps
        uint4 rr1[4], rr2[4];
        if (row_ok && full_chunk) {
          if (p.res1) {
            const uint4* r1p = reinterpret_cast<const uint4*>(p.res1 + m * p.ldr1 + col0);
#pragma unroll
            for (int k = 0; k < 4; ++k) rr1[k] = r1p[k];
          }
          if (p.res2) {
            const uint4* r2p = reinterpret_cast<const uint4*>(p.res2 + m * p.ldr2 + col0);
#pragma unroll
            for (int k = 0; k < 4; ++k) rr2[k] = r2p[k];
          }
        }
        __syncwarp();
        tmem_ld32(t_base + c, v);
        if (p.geglu) tmem_ld32(t_base + bn_out + c, gte);
        tc_wait_ld();
        float f[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) f[i] = __uint_as_float(v[i]);
        if (p.geglu) {
          float g[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) g[i] = __uint_as_float(gte[i]);
          if (p.bias) {
            if (full_chunk && ((p.N / 2) & 3) == 0) {
              const float4* bv = reinterpret_cast<const float4*>(p.bias + col0);
              const float4* bg = reinterpret_cast<const float4*>(p.bias + p.N / 2 + col0);
#pragma unroll
              for (int k = 0; k < 8; ++k) {
                const float4 x4 = __ldg(bv + k), y4 = __ldg(bg + k);
                f[4 * k] += x4.x; f[4 * k + 1] += x4.y; f[4 * k + 2] += x4.z; f[4 * k + 3] += x4.w;
                g[4 * k] += y4.x; g[4 * k + 1] += y4.y; g[4 * k + 2] += y4.z; g[4 * k + 3] += y4.w;
              }
            } else {
#pragma unroll
              for (int i = 0; i < 32; ++i) {
                if (full_chunk || col0 + i < n_out_total) {
                  f[i] += __ldg(p.bias + col0 + i);
                  g[i] += __ldg(p.bias + p.N / 2 + col0 + i);
                }
              }
            }
          }
          if (p.pre) {
            if (p.tma_store) {
              stage_store_bf16(&p.tmpre, st, lane, f, col0);
              stage_store_bf16(&p.tmpre, st, lane, g, p.N / 2 + col0);
            } else if (row_ok) {
              bf16* pv = p.pre + m * p.ldpre + col0;
              bf16* pg = pv + p.N / 2;
              if (full_chunk) {
#pragma unroll
                for (int i = 0; i < 32; i += 8) {
                  uint4 a, b;
                  a.x = pack_bf16x2(f[i], f[i + 1]); a.y = pack_bf16x2(f[i + 2], f[i + 3]);
                  a.z = pack_bf16x2(f[i + 4], f[i + 5]); a.w = pack_bf16x2(f[i + 6], f[i + 7]);
                  b.x = pack_bf16x2(g[i], g[i + 1]); b.y = pack_bf16x2(g[i + 2], g[i + 3]);
                  b.z = pack_bf16x2(g[i + 4], g[i + 5]); b.w = pack_bf16x2(g[i + 6], g[i + 7]);
                  *reinterpret_cast<uint4*>(pv + i) = a;
                  *reinterpret_cast<uint4*>(pg + i) = b;
                }
              } else {
                for (int i = 0; i < 32; ++i)
                  if (col0 + i < n_out_total) { pv[i] = __float2bfloat16(f[i]); pg[i] = __float2bfloat16(g[i]); }
              }
            }
          }
          // the reference applies GEGLU on the bf16-rounded projection (autocast F.linear output)
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const float fv = __bfloat162float(__float2bfloat16(f[i]));
            const float gv = __bfloat162float(__float2bfloat16(g[i]));
            f[i] = fv * gelu_erf_f(gv);
          }
        } else {
          if (p.bias) {
            if (full_chunk) {
              const float4* bp = reinterpret_cast<const float4*>(p.bias + col0);
#pragma unroll
              for (int k = 0; k < 8; ++k) {
                const float4 b4 = __ldg(bp + k);
                f[4 * k] += b4.x; f[4 * k + 1] += b4.y; f[4 * k + 2] += b4.z; f[4 * k + 3] += b4.w;
              }
            } else {
              for (int i = 0; i < 32; ++i)
                if (col0 + i < n_out_total) f[i] += __ldg(p.bias + col0 + i);
            }
          }
        }
        if (rb) {
          if (full_chunk && (reinterpret_cast<uintptr_t>(rb + col0) & 15) == 0) {
            const float4* bp = reinterpret_cast<const float4*>(rb + col0);
#pragma unroll
            for (int k = 0; k < 8; ++k) {
              const float4 b4 = __ldg(bp + k);
              f[4 * k] += b4.x; f[4 * k + 1] += b4.y; f[4 * k + 2] += b4.z; f[4 * k + 3] += b4.w;
            }
          } else {
#pragma unroll
            for (int i = 0; i < 32; ++i)
              if (full_chunk || col0 + i < n_out_total) f[i] += __ldg(rb + col0 + i);
          }
        }
        if (p.act) act32(f, p.act);
        if (p.scales) {
#pragma unroll
          for (int i = 0; i < 32; ++i) f[i] *= s_acc;
        }
        if (p.res1 && row_ok) {
          const bf16* r1 = p.res1 + m * p.ldr1 + col0;
          if (full_chunk) {
#pragma unroll
            for (int i = 0; i < 32; i += 8) {
              const uint4 u = rr1[i >> 3];
              float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y), c2 = unpack_bf16x2(u.z), d = unpack_bf16x2(u.w);
              f[i] += s_r1 * a.x; f[i + 1] += s_r1 * a.y; f[i + 2] += s_r1 * b.x; f[i + 3] += s_r1 * b.y;
              f[i + 4] += s_r1 * c2.x; f[i + 5] += s_r1 * c2.y; f[i + 6] += s_r1 * d.x; f[i + 7] += s_r1 * d.y;
            }
          } else {
            for (int i = 0; i < 32; ++i)
              if (col0 + i < n_out_total) f[i] += s_r1 * __bfloat162float(r1[i]);
          }
        }
        if (p.res2 && row_ok) {
          const bf16* r2 = p.res2 + m * p.ldr2 + col0;
          if (full_chunk) {
#pragma unroll
            for (int i = 0; i < 32; i += 8) {
              const uint4 u = rr2[i >> 3];
              float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y), c2 = unpack_bf16x2(u.z), d = unpack_bf16x2(u.w);
              f[i] += s_r2 * a.x; f[i + 1] += s_r2 * a.y; f[i + 2] += s_r2 * b.x; f[i + 3] += s_r2 * b.y;
              f[i + 4] += s_r2 * c2.x; f[i + 5] += s_r2 * c2.y; f[i + 6] += s_r2 * d.x; f[i + 7] += s_r2 * d.y;
            }
          } else {
            for (int i = 0; i < 32; ++i)
              if (col0 + i < n_out_total) f[i] += s_r2 * __bfloat162float(r2[i]);
          }
        }
        // ---- store
        if (p.probe == 1) {
          float acc = 0.f;
#pragma unroll
          for (int i = 0; i < 32; ++i) acc += f[i];
          if (acc == 123.456f) reinterpret_cast<float*>(p.out)[0] = acc;   // keeps the math alive
        } else if (p.tma_store) {
          if (p.out_dtype == SVDX_OUT_BF16) stage_store_bf16(&p.tmo, st, lane, f, col0);
          else stage_store_f32(&p.tmo, st, lane, f, col0, p.out_dtype == SVDX_OUT_F32_ATOMIC);
        } else if (!row_ok) {
          // nothing to write for rows past the end
        } else if (p.out_dtype == SVDX_OUT_BF16) {
          bf16* o = reinterpret_cast<bf16*>(p.out) + m * p.ldo + col0;
          if (full_chunk) {
#pragma unroll
            for (int i = 0; i < 32; i += 8) {
              uint4 a;
              a.x = pack_bf16x2(f[i], f[i + 1]); a.y = pack_bf16x2(f[i + 2], f[i + 3]);
              a.z = pack_bf16x2(f[i + 4], f[i + 5]); a.w = pack_bf16x2(f[i + 6], f[i + 7]);
              *reinterpret_cast<uint4*>(o + i) = a;
            }
          } else {
            for (int i = 0; i < 32; ++i)
              if (col0 + i < n_out_total) o[i] = __float2bfloat16(f[i]);
          }
        } else if (p.out_dtype == SVDX_OUT_F32) {
          float* o = reinterpret_cast<float*>(p.out) + m * p.ldo + col0;
          if (full_chunk) {
#pragma unroll
            for (int i = 0; i < 32; i += 4)
              *reinterpret_cast<float4*>(o + i) = make_float4(f[i], f[i + 1], f[i + 2], f[i + 3]);
          } else {
            for (int i = 0; i < 32; ++i)
              if (col0 + i < n_out_total) o[i] = f[i];
          }
        } else {
          float* o = reinterpret_cast<float*>(p.out) + m * p.ldo + col0;
          if (full_chunk) {
#pragma unroll
            for (int i = 0; i < 32; i += 4)   // 16-byte vector reductions: 4x fewer L2 atomic requests
              asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(o + i), "f"(f[i]), "f"(f[i + 1]), "f"(f[i + 2]), "f"(f[i + 3])
                           : "memory");
          } else {
            for (int i = 0; i < 32; ++i)
              if (col0 + i < n_out_total) atomicAdd(o + i, f[i]);
          }
        }
      }
}

}  // namespace svdx

// host: validates the descriptor and fills the kernel parameter block. cg = CTAs per tile (1 or 2).
int svdx_tapgemm_fill(const SvdxTapGemm* d, svdx::TapGemmKParams& p, int cg);

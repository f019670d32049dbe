// svdx_tapgemm: the tensor-core contraction of the SVD UNet hot path on sm_100a.
//
//   acc[m,n] = sum_taps sum_k A_tap[m,k] * B[n, tap*K + k]      (tcgen05.mma, fp32 accum in TMEM)
//
// One persistent, warp-specialised kernel:
//   warp 0      : TMA producer  (cp.async.bulk.tensor -> 128B-swizzled smem ring, mbarrier tx)
//   warp 1      : TMEM allocator + single-thread tcgen05.mma issuer
//   warps 2..5  : epilogue (tcgen05.ld TMEM->regs, bias/rowbias/GEGLU/residual/blend, global store)
// Accumulators are double-buffered in TMEM (2 x 256 columns) so the epilogue of tile i overlaps
// the main loop of tile i+1.
//
// A-operand modes (see include/svd_xtend_b200.h): plain/grouped rows with row-shifted taps
// (linear, (3,1,1) temporal conv [D: TemporalResnetBlock]) and channels-last images with 2-D
// shifted taps (3x3 conv [D: ResnetBlock2D/Downsample2D/Upsample2D]); zero padding comes from
// TMA out-of-bounds fill, so no im2col buffer ever exists.
#include "tapgemm_common.cuh"

namespace svdx {

template <int EPI>
__global__ void __launch_bounds__(NUM_THREADS, 1) tapgemm_kernel(const __grid_constant__ TapGemmKParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t sA = smem_base;
  const uint32_t sB = smem_base + STAGES * A_STAGE_BYTES;
  const uint32_t sEpi = sB + STAGES * B_STAGE_BYTES;   // epilogue staging (TMA stores), 4 KB per epilogue warp
  const uint32_t sBar = sEpi + NUM_EPI_WARPS * EPI_STAGE_BYTES;
  // barrier layout (8 B each): full[STAGES], empty[STAGES], tmem_full[ACC], tmem_empty[ACC], then tmem ptr
  const uint32_t bar_full = sBar;
  const uint32_t bar_empty = sBar + 8 * STAGES;
  const uint32_t bar_tfull = sBar + 16 * STAGES;
  const uint32_t bar_tempty = bar_tfull + 8 * ACC_STAGES;
  const uint32_t tmem_slot = bar_tempty + 8 * ACC_STAGES;
  uint32_t* tmem_slot_ptr = reinterpret_cast<uint32_t*>(smem_raw + (tmem_slot - smem_u32(smem_raw)));

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&p.tma);
    prefetch_tmap(&p.tmb);
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(bar_full + 8 * i, 1);
      mbar_init(bar_empty + 8 * i, 1);
    }
    for (int i = 0; i < ACC_STAGES; ++i) {
      mbar_init(bar_tfull + 8 * i, 1);
      mbar_init(bar_tempty + 8 * i, NUM_EPI_WARPS);  // one arrive per epilogue warp
    }
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, TMEM_COLS);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;

  const int total_tiles = p.m_tiles * p.n_tiles * p.split_k;
  const int b_bytes = p.block_n * BLOCK_K * 2;

  if (warp == 0) {
    // =========================== TMA producer ===========================
    const bool conv_par = (p.a_mode == SVDX_A_CONV2D) && !p.a_mn && !p.b_mn && !p.geglu && !p.wtiles && (BLOCK_M / p.W) <= 32;
    if (conv_par) {
      // warp-wide conv producer: lane 0 owns the barriers and the B tile, every lane with a row box issues it
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const int nt = tile % p.n_tiles;
        const int mt = (tile / p.n_tiles) % p.m_tiles;
        const int ks = tile / (p.n_tiles * p.m_tiles);
        const int kb0 = ks * p.kb_per_split;
        const int kb1 = min(kb0 + p.kb_per_split, p.kb_total);
        const int n0 = nt * p.block_n;
        ConvBox bx;
        conv_tile_boxes(p, mt, lane, bx);
        const CUtensorMap* amap = bx.lg == 0 ? &p.tma : &p.tma_bh[bx.lg - 1];
        int tap = kb0 / p.kb_per_tap;
        int kci = kb0 - tap * p.kb_per_tap;
        for (int kb = kb0; kb < kb1; ++kb) {
          const uint32_t full = bar_full + 8 * stage;
          if (lane == 0) {
            mbar_wait(bar_empty + 8 * stage, phase ^ 1);
            mbar_expect_tx(full, A_STAGE_BYTES + b_bytes);
          }
          __syncwarp();
          const int kc = kci * BLOCK_K;
          if (bx.active)
            tma_load_4d(amap, full, sA + stage * A_STAGE_BYTES + bx.dst_off, kc, p.tap_d0[tap], bx.hh + p.tap_d1[tap],
                        bx.nvalid ? bx.n + p.tap_d2[tap] : (1 << 28));
          if (lane == 0) tma_load_2d(&p.tmb, full, sB + stage * B_STAGE_BYTES, tap * p.K + kc, n0);
          if (++kci == p.kb_per_tap) { kci = 0; ++tap; }
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    } else if (p.a_mn && p.b_mn && p.b_mode != 1) {
      // weight-gradient forms (MN-major A and B): 2 A boxes + block_n/64 B boxes per k-block, one lane per box
      int stage = 0;
      uint32_t phase = 0;
      const int nb = p.block_n / 64;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const int nt = tile % p.n_tiles;
        const int mt = (tile / p.n_tiles) % p.m_tiles;
        const int ks = tile / (p.n_tiles * p.m_tiles);
        const int kb0 = ks * p.kb_per_split;
        const int kb1 = min(kb0 + p.kb_per_split, p.kb_total);
        const int n0 = nt * p.block_n;
        int g = 0, kbi = kb0;
        if (p.b_mode == 2) { g = kb0 / p.kb_per_group; kbi = kb0 - g * p.kb_per_group; }
        const int shift = p.b_mode == 2 ? p.tap_d0[0] : 0;
        for (int kb = kb0; kb < kb1; ++kb) {
          const uint32_t full = bar_full + 8 * stage;
          if (lane == 0) {
            mbar_wait(bar_empty + 8 * stage, phase ^ 1);
            mbar_expect_tx(full, A_STAGE_BYTES + b_bytes);
          }
          __syncwarp();
          const uint32_t dA = sA + stage * A_STAGE_BYTES;
          const uint32_t dB = sB + stage * B_STAGE_BYTES;
          if (p.b_mode == 2) {
            // group-bounded k rows (3-D maps): rows past the end of the group read as zero
            const int k0 = kbi * BLOCK_K;
            if (lane < 2) tma_load_3d(&p.tma, full, dA + lane * 8192, mt * BLOCK_M + 64 * lane, k0, g);
            else if (lane < 2 + nb) tma_load_3d(&p.tmb, full, dB + (lane - 2) * 8192, n0 + 64 * (lane - 2), k0 + shift, g);
            if (++kbi == p.kb_per_group) { kbi = 0; ++g; }
          } else {
            if (lane < 2) tma_load_2d(&p.tma, full, dA + lane * 8192, mt * BLOCK_M + 64 * lane, kb * BLOCK_K);
            else if (lane < 2 + nb) tma_load_2d(&p.tmb, full, dB + (lane - 2) * 8192, n0 + 64 * (lane - 2), kb * BLOCK_K);
          }
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    } else if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const int nt = tile % p.n_tiles;
        const int mt = (tile / p.n_tiles) % p.m_tiles;
        const int ks = tile / (p.n_tiles * p.m_tiles);
        const int kb0 = ks * p.kb_per_split;
        const int kb1 = min(kb0 + p.kb_per_split, p.kb_total);
        const int n0 = nt * (p.geglu ? p.block_n / 2 : p.block_n);
        int tap = kb0 / p.kb_per_tap;
        int kci = kb0 - tap * p.kb_per_tap - 1;
        for (int kb = kb0; kb < kb1; ++kb) {
          if (++kci == p.kb_per_tap) { kci = 0; ++tap; }   // no per-k-block division on the issue path
          mbar_wait(bar_empty + 8 * stage, phase ^ 1);
          const uint32_t full = bar_full + 8 * stage;
          mbar_expect_tx(full, A_STAGE_BYTES + b_bytes);
          const uint32_t dA = sA + stage * A_STAGE_BYTES;
          const uint32_t dB = sB + stage * B_STAGE_BYTES;
          const int kc = kci * BLOCK_K;
          // ---- A
          if (p.a_mn) {
            // memory [k rows][m cols]: two 64x64 boxes. b_mode 2 walks the k rows group by group.
            if (p.b_mode == 2) {
              // group-bounded rows (3-D map): rows past the end of the group read as zero, like the shifted B rows
              const int g = kb / p.kb_per_group;
              const int k0 = (kb - g * p.kb_per_group) * BLOCK_K;
              tma_load_3d(&p.tma, full, dA, mt * BLOCK_M, k0, g);
              tma_load_3d(&p.tma, full, dA + 8192, mt * BLOCK_M + 64, k0, g);
            } else {
              tma_load_2d(&p.tma, full, dA, mt * BLOCK_M, kb * BLOCK_K);
              tma_load_2d(&p.tma, full, dA + 8192, mt * BLOCK_M + 64, kb * BLOCK_K);
            }
          } else if (p.a_mode == SVDX_A_ROWS) {
            const int g = mt / p.tiles_per_group;
            const int t = mt - g * p.tiles_per_group;
            tma_load_3d(&p.tma, full, dA, kc, t * BLOCK_M + p.tap_d0[tap], g);
          } else if (p.wtiles) {
            // wide images (VAE encoder, W = 256 / 512): the tile is 128 consecutive pixels of one image row; the shifted
            // box (w0 + dw, h + dh) is zero-filled where it leaves the image, which IS the convolution's padding
            const int row = mt / p.wtiles;
            const int w0 = (mt - row * p.wtiles) * BLOCK_M;
            const int n = row / p.H;
            const int h = row - n * p.H;
            tma_load_4d(&p.tma, full, dA, kc, w0 + p.tap_d0[tap], h + p.tap_d1[tap], (n < p.nimg) ? n + p.tap_d2[tap] : (1 << 28));
          } else {
            // the tile's 128 pixels = R consecutive image rows; walk them image by image and cover each run with
            // the largest power-of-two row boxes available (few big TMA requests instead of R one-row requests)
            const int R = BLOCK_M / p.W;
            const int dw = p.tap_d0[tap], dh = p.tap_d1[tap], dn = p.tap_d2[tap];
            int rowid = mt * R, left = R;
            uint32_t dst = dA;
            while (left > 0) {
              const int n = rowid / p.H;
              const int h = rowid - n * p.H;
              // rows past the last image land out of bounds (n >= nimg) and are zero-filled
              const int nn = (n < p.nimg) ? n + dn : (1 << 28);
              int run = min(left, p.H - h);
              int hh = h;
              while (run > 0) {
                int lg = min(p.max_bh_log2, 31 - __clz(run));
                const int bh = 1 << lg;
                tma_load_4d(lg == 0 ? &p.tma : &p.tma_bh[lg - 1], full, dst, kc, dw, hh + dh, nn);
                dst += bh * p.W * 128;
                hh += bh; run -= bh; left -= bh; rowid += bh;
              }
            }
          }
          // ---- B
          if (p.b_mn && p.b_mode == 1) {
            // B rows are the pixels of a channels-last image tensor read at a fixed 2-D shift (conv weight gradient):
            // a k-block = 64 consecutive output pixels; out-of-image reads are zero-filled by TMA
            const int dw = p.tap_d0[0], dh = p.tap_d1[0], dn = p.tap_d2[0];
            const int pix0 = kb * BLOCK_K;
            for (int j = 0; j < p.block_n / 64; ++j) {
              if (p.W >= 64) {
                const int row = pix0 / p.W;
                const int n = row / p.H;
                const int nn = (n < p.nimg) ? n + dn : (1 << 28);
                tma_load_4d(&p.tmb, full, dB + j * 8192, n0 + 64 * j, pix0 - row * p.W + dw, row - n * p.H + dh, nn);
              } else {
                const int R = 64 / p.W;
                for (int i = 0; i < R; ++i) {
                  const int row = pix0 / p.W + i;
                  const int n = row / p.H;
                  const int nn = (n < p.nimg) ? n + dn : (1 << 28);
                  tma_load_4d(&p.tmb, full, dB + j * 8192 + i * p.W * 128, n0 + 64 * j, dw, row - n * p.H + dh, nn);
                }
              }
            }
          } else if (p.b_mn && p.b_mode == 2) {
            // B rows shifted by tap_d0[0] rows inside their group (temporal conv weight gradient)
            const int g = kb / p.kb_per_group;
            const int k0 = (kb - g * p.kb_per_group) * BLOCK_K;
            for (int j = 0; j < p.block_n / 64; ++j)
              tma_load_3d(&p.tmb, full, dB + j * 8192, n0 + 64 * j, k0 + p.tap_d0[0], g);
          } else if (p.b_mn) {
            for (int j = 0; j < p.block_n / 64; ++j)
              tma_load_2d(&p.tmb, full, dB + j * 8192, n0 + 64 * j, kb * BLOCK_K);
          } else if (p.geglu) {
            const int h = p.block_n / 2;
            tma_load_2d(&p.tmb, full, dB, tap * p.K + kc, n0);
            tma_load_2d(&p.tmb, full, dB + h * 128, tap * p.K + kc, p.N / 2 + n0);
          } else {
            tma_load_2d(&p.tmb, full, dB, tap * p.K + kc, n0);
          }
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // =========================== MMA issuer ===========================
    if (lane == 0) {
      const uint32_t idesc = make_idesc_bf16(BLOCK_M, p.block_n, p.a_mn, p.b_mn);
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        const int ks = tile / (p.n_tiles * p.m_tiles);
        const int kb0 = ks * p.kb_per_split;
        const int kb1 = min(kb0 + p.kb_per_split, p.kb_total);
        mbar_wait(bar_tempty + 8 * acc, acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * 256;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(bar_full + 8 * stage, phase);
          tc_fence_after();
          const uint32_t aaddr = sA + stage * A_STAGE_BYTES;
          const uint32_t baddr = sB + stage * B_STAGE_BYTES;
          // one descriptor per operand and stage; a 16-deep k-step advances the 16-byte start-address field
          const uint64_t ad0 = p.a_mn ? make_smem_desc_sw128(aaddr, 8192, 1024) : make_smem_desc_sw128(aaddr, 16, 1024);
          const uint64_t bd0 = p.b_mn ? make_smem_desc_sw128(baddr, 8192, 1024) : make_smem_desc_sw128(baddr, 16, 1024);
          const uint64_t astep = p.a_mn ? (2048 >> 4) : (32 >> 4), bstep = p.b_mn ? (2048 >> 4) : (32 >> 4);
#pragma unroll
          for (int j = 0; j < BLOCK_K / 16; ++j) {
            const uint64_t ad = ad0 + j * astep;
            const uint64_t bd = bd0 + j * bstep;
            umma_bf16(d_tmem, ad, bd, idesc, (kb > kb0 || j > 0) ? 1u : 0u);
          }
          umma_commit(bar_empty + 8 * stage);  // frees the smem slot when these MMAs retire
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit(bar_tfull + 8 * acc);  // accumulator complete
        if (++acc == ACC_STAGES) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else {
    // =========================== epilogue warps ===========================
    const int q = warp & 3;          // TMEM lane quarter this warp may access
    const int half = (warp - 2) >> 2;  // which of the two warps of the quarter: takes chunks half, half+2, ...
    int acc = 0;
    uint32_t acc_phase = 0;
    float s_acc = 1.f, s_r1 = 1.f, s_r2 = 1.f;
    if (p.scales) { s_acc = p.scales[0]; s_r1 = p.scales[1]; s_r2 = p.scales[2]; }
    const int n_out_total = p.geglu ? p.N / 2 : p.N;
    const int bn_out = p.geglu ? p.block_n / 2 : p.block_n;
    EpiStage st;
    st.base = sEpi + (warp - 2) * EPI_STAGE_BYTES;
    st.off = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
      const int nt = tile % p.n_tiles;
      const int mt = (tile / p.n_tiles) % p.m_tiles;
      const int n0 = nt * bn_out;
      long long m;
      bool row_ok;
      tile_row(p, mt, q * 32 + lane, m, row_ok);
      if (p.a_mode == SVDX_A_ROWS && !p.a_mn) {
        st.grp = mt / p.tiles_per_group;
        st.row0 = (mt - st.grp * p.tiles_per_group) * BLOCK_M + q * 32;
      } else {
        st.grp = 0;
        st.row0 = mt * BLOCK_M + q * 32;
      }
      // fused GroupNorm statistics: global row of this warp's first row and how many of its 32 rows exist
      long long m0;
      int valid_rows;
      if (p.a_mode == SVDX_A_ROWS && !p.a_mn) {
        m0 = (long long)st.grp * p.rows_per_group + st.row0;
        valid_rows = max(0, min(32, p.rows_per_group - st.row0));
      } else {
        m0 = st.row0;
        valid_rows = max(0, min(32, p.M - st.row0));
      }
      if constexpr (EPI == EPI_RES || EPI == EPI_RES_GN || EPI == EPI_FAST_GNB)
        prefetch_epilogue_operands(p, EPI, m0, valid_rows, n0, bn_out, n_out_total, lane, half);
      mbar_wait(bar_tfull + 8 * acc, acc_phase);
      tc_fence_after();
      const uint32_t t_base = tmem_base + acc * 256 + ((uint32_t)(q * 32) << 16);
      if constexpr (EPI == EPI_FAST || EPI == EPI_FAST_GN) epilogue_fast<EPI == EPI_FAST_GN>(p, t_base, m, row_ok, n0, half, 0, bn_out, n_out_total, st.base, st.row0, st.grp, lane, m0, valid_rows);
      else if constexpr (EPI == EPI_RES || EPI == EPI_RES_GN) epilogue_res<EPI == EPI_RES_GN>(p, t_base, m, row_ok, n0, half, 0, bn_out, n_out_total, s_acc, s_r1, s_r2, st.base, st.off, st.row0, st.grp, lane, m0, valid_rows);
      else if constexpr (EPI == EPI_GEGLU) epilogue_geglu(p, t_base, n0, half, bn_out, st.base, st.row0, st.grp, lane);
      else if constexpr (EPI == EPI_FAST_GNB) epilogue_fast_gnb(p, t_base, m, row_ok, n0, half, 0, bn_out, n_out_total, st.base, st.row0, st.grp, lane, m0, valid_rows);
      else epilogue_tile(p, t_base, m, row_ok, n0, half, bn_out, n_out_total, s_acc, s_r1, s_r2, st, lane);
      // release the accumulator stage back to the MMA warp
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_tempty + 8 * acc);
      if (++acc == ACC_STAGES) { acc = 0; acc_phase ^= 1; }
    }
    if (lane == 0) bulk_wait<0>();   // staged stores must have left shared memory (and landed) before the CTA exits
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

}  // namespace svdx

using namespace svdx;

int svdx_tapgemm_fill(const SvdxTapGemm* d, TapGemmKParams& p, int cg) {
  if (!d || !d->a || !d->b || !d->out) return svdx_fail(SVDX_E_BADARG, "tapgemm: null pointer");
  // block_n == 320: the CTA-pair kernel's two-MMA tile (256 x 320, see tapgemm2.cu) — pair-eligible problems only
  const bool wide320 = (cg == 2 && d->block_n == 320);
  if (!wide320 && (d->block_n < 32 || d->block_n > 256 || d->block_n % 32))
    return svdx_fail(SVDX_E_BADARG, "tapgemm: block_n must be a multiple of 32 in [32,256] (or 320 for CTA-pair eligible problems)");
  if (d->b_major_mn && d->block_n % 64) return svdx_fail(SVDX_E_BADARG, "tapgemm: block_n %% 64 for MN-major B");
  if (d->num_taps < 1 || d->num_taps > SVDX_MAX_TAPS) return svdx_fail(SVDX_E_BADARG, "tapgemm: num_taps");
  if (d->M <= 0 || d->N <= 0 || d->K <= 0) return svdx_fail(SVDX_E_BADARG, "tapgemm: empty problem");
  if (d->split_k < 1 || (d->split_k > 1 && d->out_dtype != SVDX_OUT_F32_ATOMIC)) return svdx_fail(SVDX_E_BADARG, "tapgemm: split_k needs atomic output");
  if (d->geglu && (d->N % 2 || d->block_n % 64 || d->b_major_mn || (d->N / 2) % (d->block_n / 2))) return svdx_fail(SVDX_E_BADARG, "tapgemm: geglu shape");
  if ((d->lda % 8) || (d->ldb % 8)) return svdx_fail(SVDX_E_BADARG, "tapgemm: lda/ldb must be multiples of 8 elements (16 B)");
  if ((reinterpret_cast<uintptr_t>(d->a) & 15) || (reinterpret_cast<uintptr_t>(d->b) & 15)) return svdx_fail(SVDX_E_BADARG, "tapgemm: operands must be 16 B aligned");
  if ((d->a_major_mn || d->b_major_mn) && (d->a_mode != SVDX_A_ROWS || d->num_taps != 1)) return svdx_fail(SVDX_E_BADARG, "tapgemm: MN-major operands only in single-tap ROWS mode");
  if (d->b_mode != 0 && !(d->a_major_mn && d->b_major_mn)) return svdx_fail(SVDX_E_BADARG, "tapgemm: b_mode needs MN-major A and B (weight-gradient form)");
  if (d->act != SVDX_ACT_NONE && (d->act != SVDX_ACT_GELU || d->geglu || d->gn_sum || d->gnb_sum || d->gnb_x || d->out_dtype != SVDX_OUT_BF16))
    return svdx_fail(SVDX_E_BADARG, "tapgemm: act needs a bf16 output and no GEGLU / gn_sum / gnb_* statistics (split-K: svdx_splitk_epilogue_act)");

  memset(&p, 0, sizeof(p));
  p.a_mode = d->a_mode; p.a_mn = d->a_major_mn; p.b_mn = d->b_major_mn;
  p.num_taps = d->num_taps;
  for (int i = 0; i < d->num_taps; ++i) { p.tap_d0[i] = d->tap_d0[i]; p.tap_d1[i] = d->tap_d1[i]; p.tap_d2[i] = d->tap_d2[i]; }
  p.M = d->M; p.N = d->N; p.K = d->K; p.block_n = d->block_n; p.split_k = d->split_k;
  p.geglu = d->geglu;
  const int bn_out = d->geglu ? d->block_n / 2 : d->block_n;
  const int n_out = d->geglu ? d->N / 2 : d->N;
  p.n_tiles = (n_out + bn_out - 1) / bn_out;

  int rc;
  p.b_mode = d->b_mode;
  if (d->a_major_mn) {
    // memory [K rows][M cols]
    if (d->groups > 1 && d->b_mode != 2) return svdx_fail(SVDX_E_BADARG, "tapgemm: MN-major A requires groups==1");
    if (d->b_mode == 2) {
      uint64_t dims[3] = {(uint64_t)d->M, (uint64_t)d->rows_per_group, (uint64_t)d->groups};
      uint64_t strides[2] = {(uint64_t)d->lda * 2, (uint64_t)d->lda * 2 * (uint64_t)d->rows_per_group};
      uint32_t box[3] = {64, 64, 1};
      rc = svdx_make_tmap(&p.tma, d->a, 3, dims, strides, box);
    } else {
      uint64_t dims[2] = {(uint64_t)d->M, (uint64_t)d->K};
      uint64_t strides[1] = {(uint64_t)d->lda * 2};
      uint32_t box[2] = {64, 64};
      rc = svdx_make_tmap(&p.tma, d->a, 2, dims, strides, box);
    }
    p.rows_per_group = d->M; p.groups = 1; p.tiles_per_group = (d->M + BLOCK_M - 1) / BLOCK_M;
    p.m_tiles = p.tiles_per_group;
  } else if (d->a_mode == SVDX_A_ROWS) {
    if (d->rows_per_group <= 0 || d->groups <= 0 || (long long)d->rows_per_group * d->groups != d->M) return svdx_fail(SVDX_E_BADARG, "tapgemm: rows_per_group*groups != M");
    uint64_t dims[3] = {(uint64_t)d->K, (uint64_t)d->rows_per_group, (uint64_t)d->groups};
    uint64_t strides[2] = {(uint64_t)d->lda * 2, (uint64_t)d->lda * 2 * (uint64_t)d->rows_per_group};
    uint32_t box[3] = {64, 128, 1};
    rc = svdx_make_tmap(&p.tma, d->a, 3, dims, strides, box);
    p.rows_per_group = d->rows_per_group; p.groups = d->groups;
    p.tiles_per_group = (d->rows_per_group + BLOCK_M - 1) / BLOCK_M;
    p.m_tiles = p.tiles_per_group * d->groups;
  } else if (d->a_mode == SVDX_A_CONV2D) {
    const bool wide = d->W > 128;
    if (d->W <= 0 || (wide ? (d->W % 128 != 0) : (128 % d->W != 0)) || d->H <= 0 || d->nimg <= 0)
      return svdx_fail(SVDX_E_BADARG, "tapgemm: conv2d needs W | 128 or 128 | W");
    // M counts output pixels of the first `M / (H*W)` images; the tensor may hold more images (parity planes)
    uint64_t dims[4] = {(uint64_t)d->K, (uint64_t)d->W, (uint64_t)d->H, (uint64_t)d->nimg};
    uint64_t strides[3] = {(uint64_t)d->lda * 2, (uint64_t)d->lda * 2 * d->W, (uint64_t)d->lda * 2 * d->W * d->H};
    uint32_t box[4] = {64, (uint32_t)(wide ? 128 : d->W), 1, 1};
    rc = svdx_make_tmap(&p.tma, d->a, 4, dims, strides, box);
    p.max_bh_log2 = 0;
    p.wtiles = wide ? d->W / 128 : 0;
    for (int lg = 1; lg <= 4 && !rc && !wide; ++lg) {
      const int bh = 1 << lg;
      if (bh * d->W > BLOCK_M || bh > d->H) break;
      uint32_t boxh[4] = {64, (uint32_t)d->W, (uint32_t)bh, 1};
      rc = svdx_make_tmap(&p.tma_bh[lg - 1], d->a, 4, dims, strides, boxh);
      p.max_bh_log2 = lg;
    }
    p.W = d->W; p.H = d->H; p.nimg = d->M / (d->H * d->W);
    if ((long long)p.nimg * d->H * d->W != d->M) return svdx_fail(SVDX_E_BADARG, "tapgemm: conv2d M must be images*H*W");
    p.m_tiles = (d->M + BLOCK_M - 1) / BLOCK_M;
    p.rows_per_group = d->M; p.groups = 1; p.tiles_per_group = p.m_tiles;
  } else {
    return svdx_fail(SVDX_E_BADARG, "tapgemm: a_mode");
  }
  if (rc) return rc;

  if (d->b_major_mn && d->b_mode == 1) {
    if (d->W <= 0 || d->H <= 0 || d->nimg <= 0 || (d->W < 64 && 64 % d->W) || (d->W >= 64 && d->W % 64)) return svdx_fail(SVDX_E_BADARG, "tapgemm: b_mode 1 needs W | 64 or 64 | W");
    uint64_t dims[4] = {(uint64_t)d->N, (uint64_t)d->W, (uint64_t)d->H, (uint64_t)d->nimg};
    uint64_t strides[3] = {(uint64_t)d->ldb * 2, (uint64_t)d->ldb * 2 * d->W, (uint64_t)d->ldb * 2 * d->W * d->H};
    uint32_t box[4] = {64, (uint32_t)(d->W >= 64 ? 64 : d->W), 1, 1};
    rc = svdx_make_tmap(&p.tmb, d->b, 4, dims, strides, box);
    p.W = d->W; p.H = d->H; p.nimg = d->K / (d->W * d->H);   // K = output pixels = images * H * W
    if ((long long)p.nimg * d->W * d->H != d->K) return svdx_fail(SVDX_E_BADARG, "tapgemm: b_mode 1 K must be images*H*W");
  } else if (d->b_major_mn && d->b_mode == 2) {
    if (d->rows_per_group <= 0 || d->groups <= 0 || (long long)d->rows_per_group * d->groups != d->K) return svdx_fail(SVDX_E_BADARG, "tapgemm: b_mode 2 rows_per_group*groups != K");
    uint64_t dims[3] = {(uint64_t)d->N, (uint64_t)d->rows_per_group, (uint64_t)d->groups};
    uint64_t strides[2] = {(uint64_t)d->ldb * 2, (uint64_t)d->ldb * 2 * (uint64_t)d->rows_per_group};
    uint32_t box[3] = {64, 64, 1};
    rc = svdx_make_tmap(&p.tmb, d->b, 3, dims, strides, box);
    p.rows_per_group = d->rows_per_group; p.groups = d->groups;
  } else if (d->b_major_mn) {
    uint64_t dims[2] = {(uint64_t)d->N, (uint64_t)d->K};
    uint64_t strides[1] = {(uint64_t)d->ldb * 2};
    uint32_t box[2] = {64, 64};
    rc = svdx_make_tmap(&p.tmb, d->b, 2, dims, strides, box);
  } else {
    uint64_t dims[2] = {(uint64_t)d->K * d->num_taps, (uint64_t)d->N};
    uint64_t strides[1] = {(uint64_t)d->ldb * 2};
    // a CTA of a pair fetches half of the B tile; a GEGLU tile is already fetched as two halves (value | gate)
    uint32_t box[2] = {64, (uint32_t)(wide320 ? 80 : (d->geglu || cg == 2) ? d->block_n / 2 : d->block_n)};
    rc = svdx_make_tmap(&p.tmb, d->b, 2, dims, strides, box);
  }
  if (rc) return rc;
  p.tiles_per_group_pairs = (p.tiles_per_group + 1) / 2;
  p.pair_m_tiles = p.tiles_per_group_pairs * p.groups;

  p.kb_per_tap = (d->K + BLOCK_K - 1) / BLOCK_K;
  p.kb_total = p.kb_per_tap * d->num_taps;
  p.kb_per_group = p.kb_per_tap;
  if (d->b_mode == 2) {
    p.kb_per_group = (d->rows_per_group + BLOCK_K - 1) / BLOCK_K;
    p.kb_per_tap = p.kb_per_group * d->groups;
    p.kb_total = p.kb_per_tap;
  }
  p.kb_per_split = (p.kb_total + d->split_k - 1) / d->split_k;
  // drop empty splits
  p.split_k = (p.kb_total + p.kb_per_split - 1) / p.kb_per_split;

  p.out = d->out; p.ldo = d->ldo; p.out_dtype = d->out_dtype;
  p.bias = d->bias; p.rowbias = d->rowbias; p.rowbias_div = d->rowbias_div > 0 ? d->rowbias_div : 1; p.ldrb = d->ldrb;
  p.res1 = reinterpret_cast<const bf16*>(d->res1); p.ldr1 = d->ldr1;
  p.res2 = reinterpret_cast<const bf16*>(d->res2); p.ldr2 = d->ldr2;
  p.scales = d->scales; p.pre = reinterpret_cast<bf16*>(d->pre); p.ldpre = d->ldpre;
  p.gn_sum = d->gn_sum; p.gn_ld = d->gn_ld; p.gn_rows = d->gn_rows;
  p.gnb_x = reinterpret_cast<const bf16*>(d->gnb_x); p.gnb_ldx = d->gnb_ldx; p.gnb_c1 = d->gnb_x2 ? d->gnb_c1 : d->N;
  p.gnb_x2 = reinterpret_cast<const bf16*>(d->gnb_x2); p.gnb_ldx2 = d->gnb_ldx2;
  p.gnb_ab = d->gnb_ab; p.gnb_sum = d->gnb_sum; p.gnb_rows = d->gnb_rows; p.gnb_silu = d->gnb_silu;
  p.act = d->act;
  {
    static int probe = -1;
    if (probe < 0) { const char* e = getenv("SVDX_EPI_PROBE"); probe = e ? atoi(e) : 0; }
    p.probe = probe;
  }
  // staged TMA stores: the output as a {columns, rows-per-group, groups} tensor so that ragged last tiles are clipped
  {
    static int use = -1;
    if (use < 0) { const char* e = getenv("SVDX_TMA_STORE"); use = e ? atoi(e) : 1; }
    const bool grouped = (d->a_mode == SVDX_A_ROWS && !d->a_major_mn);
    const uint64_t R = grouped ? (uint64_t)d->rows_per_group : (uint64_t)d->M;
    const uint64_t G = grouped ? (uint64_t)d->groups : 1;
    const bool f32 = d->out_dtype != SVDX_OUT_BF16;
    const int esz = f32 ? 4 : 2;
    bool ok = use != 0 && (d->ldo * esz) % 16 == 0 && (reinterpret_cast<uintptr_t>(d->out) & 15) == 0;
    if (d->geglu && d->pre && ((d->N / 2) % 32 || (d->ldpre % 8) || (reinterpret_cast<uintptr_t>(d->pre) & 15))) ok = false;
    if (ok) {
      uint64_t dims[3] = {(uint64_t)n_out, R, G};
      uint64_t strides[2] = {(uint64_t)d->ldo * esz, (uint64_t)d->ldo * esz * R};
      uint32_t box[3] = {32, 32, 1};
      rc = svdx_make_tmap_ex(&p.tmo, d->out, f32, f32 ? 128 : 64, 3, dims, strides, box);
      if (rc) return rc;
      if (d->geglu && d->pre) {
        uint64_t pdims[3] = {(uint64_t)d->N, R, G};
        uint64_t pstrides[2] = {(uint64_t)d->ldpre * 2, (uint64_t)d->ldpre * 2 * R};
        rc = svdx_make_tmap_ex(&p.tmpre, d->pre, 0, 64, 3, pdims, pstrides, box);
        if (rc) return rc;
      }
      p.tma_store = 1;
    }
    // specialised epilogues: bf16 through TMA, whole 32-column chunks, 16-byte aligned bias rows
    p.epi_mode = EPI_GENERIC;
    const bool vec_ok = (reinterpret_cast<uintptr_t>(d->bias) & 15) == 0
                        && (!d->rowbias || ((reinterpret_cast<uintptr_t>(d->rowbias) & 15) == 0 && d->ldrb % 4 == 0));
    if (p.tma_store && !f32 && n_out % 32 == 0 && vec_ok && !p.probe && use != 2)
      p.epi_mode = d->geglu ? EPI_GEGLU : (d->res1 || d->res2 || d->scales) ? EPI_RES : EPI_FAST;
  }
  if (p.split_k > 1 && (p.bias || p.rowbias || p.res1 || p.res2 || p.geglu)) return svdx_fail(SVDX_E_BADARG, "tapgemm: split_k with epilogue operands");
  if (p.gnb_sum) {
    if (p.epi_mode != EPI_FAST || p.gn_sum)
      return svdx_fail(SVDX_E_BADARG, "tapgemm: gnb_sum needs the plain bf16 TMA-store epilogue (no residual / scales / GEGLU / split-K / gn_sum)");
    if (!p.gnb_x || p.gnb_rows <= 0 || (p.gnb_silu && !p.gnb_ab) || (d->N & 1) || (p.gnb_ldx % 8) || (reinterpret_cast<uintptr_t>(p.gnb_x) & 15) ||
        (reinterpret_cast<uintptr_t>(p.gnb_sum) & 7) || (p.gnb_ab && (reinterpret_cast<uintptr_t>(p.gnb_ab) & 7)) ||
        (p.gnb_x2 && (p.gnb_c1 <= 0 || p.gnb_c1 >= d->N || p.gnb_c1 % 32 || (p.gnb_ldx2 % 8) || (reinterpret_cast<uintptr_t>(p.gnb_x2) & 15))))
      return svdx_fail(SVDX_E_BADARG, "tapgemm: gnb operands (x rows 16-byte aligned, gnb_rows > 0, scale/shift table for SiLU, concat split % 32)");
    p.epi_mode = EPI_FAST_GNB;
  }
  if (wide320 && p.epi_mode != EPI_FAST && p.epi_mode != EPI_RES && p.epi_mode != EPI_FAST_GNB)
    return svdx_fail(SVDX_E_BADARG, "tapgemm: block_n 320 needs a bf16 output through the TMA-store epilogues (N % 320 == 0, aligned rows)");
  if (p.gn_sum) {
    if (p.epi_mode != EPI_FAST && p.epi_mode != EPI_RES)
      return svdx_fail(SVDX_E_BADARG, "tapgemm: gn_sum needs a bf16 output through the TMA-store epilogues (N % 32 == 0, aligned rows), no split-K / GEGLU");
    if (p.gn_rows <= 0 || p.gn_ld < n_out || (p.gn_ld & 1) || (reinterpret_cast<uintptr_t>(p.gn_sum) & 7))
      return svdx_fail(SVDX_E_BADARG, "tapgemm: gn_sum needs gn_rows > 0, even gn_ld >= N, 8-byte aligned buffer");
  }
  // vector paths need 16 B alignment of every row start
  if (d->out_dtype == SVDX_OUT_BF16 && ((d->ldo % 8) || (reinterpret_cast<uintptr_t>(d->out) & 15))) return svdx_fail(SVDX_E_BADARG, "tapgemm: out alignment");
  if (d->out_dtype != SVDX_OUT_BF16 && ((d->ldo % 4) || (reinterpret_cast<uintptr_t>(d->out) & 15))) return svdx_fail(SVDX_E_BADARG, "tapgemm: out alignment");
  if (d->res1 && ((d->ldr1 % 8) || (reinterpret_cast<uintptr_t>(d->res1) & 15))) return svdx_fail(SVDX_E_BADARG, "tapgemm: res1 alignment");
  if (d->res2 && ((d->ldr2 % 8) || (reinterpret_cast<uintptr_t>(d->res2) & 15))) return svdx_fail(SVDX_E_BADARG, "tapgemm: res2 alignment");
  if (d->pre && ((d->ldpre % 8) || (reinterpret_cast<uintptr_t>(d->pre) & 15))) return svdx_fail(SVDX_E_BADARG, "tapgemm: pre alignment");

  return SVDX_OK;
}

int svdx_tapgemm2_launch(const TapGemmKParams& p, cudaStream_t stream);   // tapgemm2.cu
bool svdx_tapgemm2_eligible(const SvdxTapGemm* d);

extern "C" int svdx_tapgemm(const SvdxTapGemm* d, void* stream_v) {
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_v);
  TapGemmKParams p;
  const bool pair = svdx_tapgemm2_eligible(d);
  int rc = svdx_tapgemm_fill(d, p, pair ? 2 : 1);
  if (rc) return rc;
  if (pair) return svdx_tapgemm2_launch(p, stream);
  static bool attr_done[SVDX_MAX_DEVICES] = {false};
  const int slot = svdx_device_slot();
  if (!attr_done[slot]) {
    cudaError_t e = cudaFuncSetAttribute(tapgemm_kernel<EPI_GENERIC>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(tapgemm_kernel<EPI_FAST>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(tapgemm_kernel<EPI_GEGLU>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(tapgemm_kernel<EPI_RES>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(tapgemm_kernel<EPI_FAST_GN>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(tapgemm_kernel<EPI_RES_GN>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(tapgemm_kernel<EPI_FAST_GNB>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
    if (e != cudaSuccess) return svdx_fail_cuda(e, "tapgemm: set smem attribute");
    attr_done[slot] = true;
  }
  const int total_tiles = p.m_tiles * p.n_tiles * p.split_k;
  int grid = svdx_num_sms();
  if (grid > total_tiles) grid = total_tiles;
  if (p.epi_mode == EPI_FAST_GNB) tapgemm_kernel<EPI_FAST_GNB><<<grid, NUM_THREADS, SMEM_BYTES, stream>>>(p);
  else if (p.epi_mode == EPI_FAST && p.gn_sum) tapgemm_kernel<EPI_FAST_GN><<<grid, NUM_THREADS, SMEM_BYTES, stream>>>(p);
  else if (p.epi_mode == EPI_RES && p.gn_sum) tapgemm_kernel<EPI_RES_GN><<<grid, NUM_THREADS, SMEM_BYTES, stream>>>(p);
  else if (p.epi_mode == EPI_FAST) tapgemm_kernel<EPI_FAST><<<grid, NUM_THREADS, SMEM_BYTES, stream>>>(p);
  else if (p.epi_mode == EPI_GEGLU) tapgemm_kernel<EPI_GEGLU><<<grid, NUM_THREADS, SMEM_BYTES, stream>>>(p);
  else if (p.epi_mode == EPI_RES) tapgemm_kernel<EPI_RES><<<grid, NUM_THREADS, SMEM_BYTES, stream>>>(p);
  else tapgemm_kernel<EPI_GENERIC><<<grid, NUM_THREADS, SMEM_BYTES, stream>>>(p);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return svdx_fail_cuda(e, "tapgemm: launch");
  return SVDX_OK;
}

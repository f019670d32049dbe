// ViT self-attention of the CLIP image encoder (transformers CLIPAttention of CLIPVisionModelWithProjection, train_svd.py:646,
// :875): head_dim 80, no mask, one sequence of S <= 512 tokens per image (257 = 16 x 16 patches + the class token), forward only.
//
// Why not the tcgen05 kernel of attention.cu: it is specialised to head_dim 64 and 128-row tiles; 257 tokens fill 3 such tiles
// at 67 % padding, and the whole op is small (2 x 257 x 257 x 80 x 2 x 16 heads = 0.34 GFLOP per layer at B = 1, ~1 % of the
// layer's linears). The form below follows attention_small.cu: warp-level tensor-core MMAs (mma.sync m16n8k16, bf16 -> fp32)
// with the whole K / V head slice of the sequence resident in shared memory.
//   * one CTA per (image, head, 64-query block), 4 warps x 16 query rows: 5 x 16 x B CTAs (80 at B = 1);
//   * K, V (S x 80, zero rows past S) and the CTA's 64 Q rows are staged with cp.async into rows of 88 bf16 (176 B: 16-byte
//     aligned rows, conflict-free 32-bit fragment loads and ldmatrix.trans);
//   * keys are consumed in 64-key chunks with an online softmax (running row max / sum in the log2 domain); the ragged tail
//     (257 = 4 x 64 + 1) is masked to -inf, every chunk holds at least one valid key so the running max stays finite;
//   * the output goes back through the warp's (no longer needed) Q rows as full 16-byte stores.
// q, k and v are read in place from the fused [tokens][3C] q|k|v matrix (head h at columns h * 80: 160-byte offsets).
#include "common.cuh"
#include "../../include/svd_xtend_b200.h"
#include "host_util.h"

namespace svdx {

constexpr int VIT_D = 80;
constexpr int VIT_ROW = 88;        // staged row: 80 + 8 pad bf16
constexpr int VIT_WARPS = 4;
constexpr int VIT_QB = 16 * VIT_WARPS;
constexpr int VIT_KC = 64;         // keys per online-softmax chunk
constexpr int VIT_MAX_S = 512;
constexpr float VIT_LOG2E = 1.4426950408889634f;

struct VitAttnP {
  const bf16 *q, *k, *v;
  bf16* out;
  long long ldq, ldk, ldv, ldo, seq_stride;
  int S, Sp;
  float scale;
};

SVDX_DEVINL void vit_mma(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
SVDX_DEVINL uint32_t vit_lds32(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}
SVDX_DEVINL void cp_async16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}

// rows [0, nrows) of a [*, 80] head slice -> staged rows; rows in [nrows, rows_alloc) are zero
SVDX_DEVINL void vit_stage(const bf16* __restrict__ src, long long ld, int nrows, int rows_alloc, uint32_t tile) {
  for (int i = threadIdx.x; i < rows_alloc * (VIT_D / 8); i += blockDim.x) {
    const int r = i / (VIT_D / 8), c = i - r * (VIT_D / 8);
    const uint32_t dst = tile + (uint32_t)(r * VIT_ROW + c * 8) * 2u;
    if (r < nrows) cp_async16(dst, src + (long long)r * ld + c * 8);
    else st_shared_v4(dst, 0u, 0u, 0u, 0u);
  }
}

__global__ void __launch_bounds__(VIT_WARPS * 32) attn_vit_fwd_kernel(const VitAttnP p) {
  extern __shared__ __align__(16) uint8_t vs_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, tq = lane & 3;
  const int qb = blockIdx.x, h = blockIdx.y;
  const long long tok0 = (long long)blockIdx.z * p.seq_stride;
  const int S = p.S, Sp = p.Sp;
  const int q0 = qb * VIT_QB;
  const uint32_t tK = smem_u32(vs_smem), tV = tK + (uint32_t)Sp * VIT_ROW * 2u, tQ = tV + (uint32_t)Sp * VIT_ROW * 2u;

  vit_stage(p.q + (tok0 + q0) * p.ldq + h * VIT_D, p.ldq, min(VIT_QB, S - q0), VIT_QB, tQ);
  vit_stage(p.k + tok0 * p.ldk + h * VIT_D, p.ldk, S, Sp, tK);
  vit_stage(p.v + tok0 * p.ldv + h * VIT_D, p.ldv, S, Sp, tV);
  asm volatile("cp.async.commit_group;" ::: "memory");
  asm volatile("cp.async.wait_group 0;" ::: "memory");
  __syncthreads();

  // Q fragments of this warp's 16 rows (A operand, 5 k-steps of 16 head dims)
  const uint32_t tQw = tQ + (uint32_t)(warp * 16) * VIT_ROW * 2u;
  uint32_t qa[5][4];
#pragma unroll
  for (int ks = 0; ks < 5; ++ks) {
    const uint32_t base = tQw + (uint32_t)(g * VIT_ROW + ks * 16 + 2 * tq) * 2u;
    qa[ks][0] = vit_lds32(base);
    qa[ks][1] = vit_lds32(base + 8 * VIT_ROW * 2);
    qa[ks][2] = vit_lds32(base + 16);
    qa[ks][3] = vit_lds32(base + 8 * VIT_ROW * 2 + 16);
  }
  const float qs = p.scale * VIT_LOG2E;
  float o[10][4];
#pragma unroll
  for (int dn = 0; dn < 10; ++dn)
#pragma unroll
    for (int i = 0; i < 4; ++i) o[dn][i] = 0.f;
  float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;   // rows g and g + 8: running max (log2 domain), partial sums

#pragma unroll 1
  for (int kc = 0; kc < Sp; kc += VIT_KC) {
    float s[8][4];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt)
#pragma unroll
      for (int i = 0; i < 4; ++i) s[nt][i] = 0.f;
#pragma unroll
    for (int ks = 0; ks < 5; ++ks) {
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        const uint32_t base = tK + (uint32_t)((kc + nt * 8 + g) * VIT_ROW + ks * 16 + 2 * tq) * 2u;
        vit_mma(s[nt], qa[ks], vit_lds32(base), vit_lds32(base + 16));
      }
    }
    float mx0 = m0, mx1 = m1;
#pragma unroll
    for (int nt = 0; nt < 8; ++nt)
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        const bool ok = kc + nt * 8 + 2 * tq + i < S;
        s[nt][i] = ok ? s[nt][i] * qs : -INFINITY;
        s[nt][2 + i] = ok ? s[nt][2 + i] * qs : -INFINITY;
        mx0 = fmaxf(mx0, s[nt][i]);
        mx1 = fmaxf(mx1, s[nt][2 + i]);
      }
    mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
    mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
    mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
    mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
    const float c0 = exp2_fast(m0 - mx0), c1 = exp2_fast(m1 - mx1);   // first chunk: exp2(-inf) = 0
    m0 = mx0; m1 = mx1;
    l0 *= c0; l1 *= c1;
#pragma unroll
    for (int dn = 0; dn < 10; ++dn) { o[dn][0] *= c0; o[dn][1] *= c0; o[dn][2] *= c1; o[dn][3] *= c1; }
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      s[nt][0] = exp2_fast(s[nt][0] - mx0); s[nt][1] = exp2_fast(s[nt][1] - mx0);
      s[nt][2] = exp2_fast(s[nt][2] - mx1); s[nt][3] = exp2_fast(s[nt][3] - mx1);
      l0 += s[nt][0] + s[nt][1];
      l1 += s[nt][2] + s[nt][3];
    }
    // O += P V: the score accumulator layout is the A-operand layout of the next MMA; V rows through ldmatrix.trans
#pragma unroll
    for (int kk = 0; kk < VIT_KC / 16; ++kk) {
      uint32_t a[4];
      a[0] = pack_bf16x2(s[2 * kk][0], s[2 * kk][1]);
      a[1] = pack_bf16x2(s[2 * kk][2], s[2 * kk][3]);
      a[2] = pack_bf16x2(s[2 * kk + 1][0], s[2 * kk + 1][1]);
      a[3] = pack_bf16x2(s[2 * kk + 1][2], s[2 * kk + 1][3]);
#pragma unroll
      for (int dn = 0; dn < 10; ++dn) {
        uint32_t b0, b1;
        const uint32_t addr = tV + (uint32_t)((kc + kk * 16 + (lane & 15)) * VIT_ROW + dn * 8) * 2u;
        asm volatile("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0, %1}, [%2];" : "=r"(b0), "=r"(b1) : "r"(addr));
        vit_mma(o[dn], a, b0, b1);
      }
    }
  }
  l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
  l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
  const float i0 = 1.0f / l0, i1 = 1.0f / l1;
  // the warp's Q rows are free (fragments are in registers): stage the 16 output rows there
  __syncwarp();
#pragma unroll
  for (int dn = 0; dn < 10; ++dn) {
    const uint32_t base = tQw + (uint32_t)(g * VIT_ROW + dn * 8 + 2 * tq) * 2u;
    asm volatile("st.shared.b32 [%0], %1;" ::"r"(base), "r"(pack_bf16x2(o[dn][0] * i0, o[dn][1] * i0)) : "memory");
    asm volatile("st.shared.b32 [%0], %1;" ::"r"(base + 8 * VIT_ROW * 2), "r"(pack_bf16x2(o[dn][2] * i1, o[dn][3] * i1)) : "memory");
  }
  __syncwarp();
  const int r0 = q0 + warp * 16;
  bf16* dst = p.out + (tok0 + r0) * p.ldo + h * VIT_D;
#pragma unroll
  for (int it = 0; it < 5; ++it) {
    const int i = it * 32 + lane;
    const int r = i / 10, c = i - r * 10;
    if (r0 + r < S) {
      uint4 u;
      asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(u.x), "=r"(u.y), "=r"(u.z), "=r"(u.w) : "r"(tQw + (uint32_t)(r * VIT_ROW + c * 8) * 2u));
      *reinterpret_cast<uint4*>(dst + (long long)r * p.ldo + c * 8) = u;
    }
  }
}

}  // namespace svdx

using namespace svdx;

extern "C" int svdx_attention_vit_fwd(const SvdxAttn* d, void* stream) {
  if (!d || !d->q || !d->k || !d->v || !d->o) return svdx_fail(SVDX_E_BADARG, "attention_vit: null pointer");
  if (d->S < 1 || d->S > VIT_MAX_S) return svdx_fail(SVDX_E_BADARG, "attention_vit: S must be in [1, 512]");
  if (d->heads <= 0 || d->heads > 65535 || d->nseq <= 0 || d->nseq > 65535 || d->inner != 1 || d->tok_stride != 1 || d->outer_stride < d->S)
    return svdx_fail(SVDX_E_BADARG, "attention_vit: sequences must be contiguous blocks of S rows (inner = 1, tok_stride = 1, outer_stride >= S)");
  if ((d->ldq % 8) || (d->ldk % 8) || (d->ldv % 8) || (d->ldo % 8)) return svdx_fail(SVDX_E_BADARG, "attention_vit: leading dims must be multiples of 8");
  if (d->ldq < (long long)d->heads * VIT_D || d->ldk < (long long)d->heads * VIT_D || d->ldv < (long long)d->heads * VIT_D || d->ldo < (long long)d->heads * VIT_D)
    return svdx_fail(SVDX_E_BADARG, "attention_vit: leading dims must hold heads * 80 columns");
  const uintptr_t al = reinterpret_cast<uintptr_t>(d->q) | reinterpret_cast<uintptr_t>(d->k) | reinterpret_cast<uintptr_t>(d->v) | reinterpret_cast<uintptr_t>(d->o);
  if (al & 15) return svdx_fail(SVDX_E_BADARG, "attention_vit: operands must be 16 B aligned");
  VitAttnP p;
  p.q = reinterpret_cast<const bf16*>(d->q); p.k = reinterpret_cast<const bf16*>(d->k); p.v = reinterpret_cast<const bf16*>(d->v);
  p.out = reinterpret_cast<bf16*>(d->o);
  p.ldq = d->ldq; p.ldk = d->ldk; p.ldv = d->ldv; p.ldo = d->ldo; p.seq_stride = d->outer_stride;
  p.S = d->S;
  p.Sp = (d->S + VIT_KC - 1) / VIT_KC * VIT_KC;
  p.scale = d->scale;
  const size_t smem = (size_t)(2 * p.Sp + VIT_QB) * VIT_ROW * 2;
  static bool attr_done[SVDX_MAX_DEVICES] = {false};
  const int slot = svdx_device_slot();
  if (!attr_done[slot]) {
    cudaError_t e = cudaFuncSetAttribute(attn_vit_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (2 * VIT_MAX_S + VIT_QB) * VIT_ROW * 2);
    if (e != cudaSuccess) return svdx_fail_cuda(e, "attention_vit: set smem attribute");
    attr_done[slot] = true;
  }
  const dim3 grid((unsigned)((d->S + VIT_QB - 1) / VIT_QB), (unsigned)d->heads, (unsigned)d->nseq);
  attn_vit_fwd_kernel<<<grid, VIT_WARPS * 32, smem, reinterpret_cast<cudaStream_t>(stream)>>>(p);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return svdx_fail_cuda(e, "attention_vit: launch");
  return SVDX_OK;
}

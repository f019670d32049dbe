// Elementwise / layout / reduction kernels of the SVD UNet hot path (HBM-bound, CUDA cores):
// weight preparation (fp32 master -> bf16 operand layouts), NCHW<->channels-last boundary
// conversion, nearest-2x upsample, stride-2 parity planes, channel concat/split, GEGLU backward,
// bias-gradient column sums, AlphaBlender scales, fused AdamW.
// All 16-byte vectorised where the layout allows; grids are sized from the element count.
#include "common.cuh"
#include "../../include/svd_xtend_b200.h"
#include "host_util.h"
#include <cuda_fp16.h>
#include <type_traits>

namespace svdx {

SVDX_DEVINL long long gtid() { return (long long)blockIdx.x * blockDim.x + threadIdx.x; }
static inline unsigned nblocks(long long n, int threads = 256) { return (unsigned)((n + threads - 1) / threads); }

// ------------------------------------------------------------------ weight prep
template <typename T>
SVDX_DEVINL float ldf(const T* p, long long i);
template <>
SVDX_DEVINL float ldf<float>(const float* p, long long i) { return p[i]; }
template <>
SVDX_DEVINL float ldf<bf16>(const bf16* p, long long i) { return __bfloat162float(p[i]); }
template <>
SVDX_DEVINL float ldf<__half>(const __half* p, long long i) { return __half2float(p[i]); }

// mode 0: dst[o][i]            = src[o][i]          (taps == 1)
// mode 2: dst[o][t][i_pad]     = src[o][i][t]
// mode 3: dst[i][t][o]         = src[o][i][t]
template <typename T>
__global__ void prep_gather_kernel(const T* __restrict__ src, bf16* __restrict__ dst, int mode, int O, int I, int taps, int i_pad) {
  const long long idx = gtid();
  if (mode == 0) {
    if (idx >= (long long)O * I) return;
    dst[idx] = __float2bfloat16(ldf(src, idx));
  } else if (mode == 2) {
    const long long total = (long long)O * taps * i_pad;
    if (idx >= total) return;
    const int i = (int)(idx % i_pad);
    const int t = (int)((idx / i_pad) % taps);
    const int o = (int)(idx / ((long long)i_pad * taps));
    dst[idx] = (i < I) ? __float2bfloat16(ldf(src, ((long long)o * I + i) * taps + t)) : __float2bfloat16(0.f);
  } else {
    const long long total = (long long)I * taps * O;
    if (idx >= total) return;
    const int o = (int)(idx % O);
    const int t = (int)((idx / O) % taps);
    const int i = (int)(idx / ((long long)O * taps));
    dst[idx] = __float2bfloat16(ldf(src, ((long long)o * I + i) * taps + t));
  }
}

// mode 1: dst[i][o] = src[o][i]  — 32x32 shared-memory tile transpose
template <typename T>
__global__ void prep_transpose_kernel(const T* __restrict__ src, bf16* __restrict__ dst, int O, int I) {
  __shared__ float tile[32][33];
  const int i0 = blockIdx.x * 32, o0 = blockIdx.y * 32;
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const int o = o0 + r, i = i0 + threadIdx.x;
    tile[r][threadIdx.x] = (o < O && i < I) ? ldf(src, (long long)o * I + i) : 0.f;
  }
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {
    const int i = i0 + r, o = o0 + threadIdx.x;
    if (i < I && o < O) dst[(long long)i * O + o] = __float2bfloat16(tile[threadIdx.x][r]);
  }
}

__global__ void cast_f32_bf16_kernel(const float* __restrict__ src, bf16* __restrict__ dst, long long n) {
  const long long i = gtid() * 4;
  if (i + 3 < n) {
    const float4 v = *reinterpret_cast<const float4*>(src + i);
    uint2 o;
    o.x = pack_bf16x2(v.x, v.y);
    o.y = pack_bf16x2(v.z, v.w);
    *reinterpret_cast<uint2*>(dst + i) = o;
  } else {
    for (long long k = i; k < n; ++k) dst[k] = __float2bfloat16(src[k]);
  }
}
__global__ void cast_bf16_f32_kernel(const bf16* __restrict__ src, float* __restrict__ dst, long long n) {
  const long long i = gtid();
  if (i < n) dst[i] = __bfloat162float(src[i]);
}
__global__ void cast_f16_f32_kernel(const __half* __restrict__ src, float* __restrict__ dst, long long n) {
  const long long i = gtid();
  if (i < n) dst[i] = __half2float(src[i]);
}

// ------------------------------------------------------------------ layout boundary
template <typename T>
__global__ void nchw_to_nhwc_kernel(const T* __restrict__ src, bf16* __restrict__ dst, int N, int C, int H, int W, int c_pad) {
  const long long idx = gtid();
  const long long total = (long long)N * H * W * c_pad;
  if (idx >= total) return;
  const int c = (int)(idx % c_pad);
  const long long pix = idx / c_pad;
  const int w = (int)(pix % W);
  const int h = (int)((pix / W) % H);
  const int n = (int)(pix / ((long long)W * H));
  dst[idx] = (c < C) ? __float2bfloat16(ldf(src, (((long long)n * C + c) * H + h) * W + w)) : __float2bfloat16(0.f);
}
template <typename T>
__global__ void nhwc_to_nchw_kernel(const bf16* __restrict__ src, long long lds, T* __restrict__ dst, int N, int C, int H, int W) {
  const long long idx = gtid();
  const long long total = (long long)N * C * H * W;
  if (idx >= total) return;
  const int w = (int)(idx % W);
  const int h = (int)((idx / W) % H);
  const int c = (int)((idx / ((long long)W * H)) % C);
  const int n = (int)(idx / ((long long)W * H * C));
  const float v = __bfloat162float(src[(((long long)n * H + h) * W + w) * lds + c]);
  if constexpr (sizeof(T) == 4) dst[idx] = v;
  else if constexpr (std::is_same<T, __half>::value) dst[idx] = __float2half(v);
  else dst[idx] = __float2bfloat16(v);
}

// nearest 2x: dst[n][2h+a][2w+b][:] = src[n][h][w][:]   (16 B vectors)
__global__ void upsample2x_kernel(const uint4* __restrict__ src, uint4* __restrict__ dst, int N, int H, int W, int CV) {
  const long long idx = gtid();
  const long long total = (long long)N * 2 * H * 2 * W * CV;
  if (idx >= total) return;
  const int cv = (int)(idx % CV);
  const long long pix = idx / CV;
  const int w2 = (int)(pix % (2 * W));
  const int h2 = (int)((pix / (2 * W)) % (2 * H));
  const int n = (int)(pix / ((long long)4 * W * H));
  dst[idx] = src[(((long long)n * H + (h2 >> 1)) * W + (w2 >> 1)) * CV + cv];
}
SVDX_DEVINL uint32_t add_bf16x2_f32(uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  const float2 x = unpack_bf16x2(a), y = unpack_bf16x2(b), z = unpack_bf16x2(c), w = unpack_bf16x2(d);
  return pack_bf16x2(x.x + y.x + z.x + w.x, x.y + y.y + z.y + w.y);
}
// adjoint: ddst[n][h][w] = sum of the 2x2 block of dsrc
__global__ void upsample2x_bwd_kernel(const uint4* __restrict__ dsrc, uint4* __restrict__ ddst, int N, int H, int W, int CV) {
  const long long idx = gtid();
  const long long total = (long long)N * H * W * CV;
  if (idx >= total) return;
  const int cv = (int)(idx % CV);
  const long long pix = idx / CV;
  const int w = (int)(pix % W);
  const int h = (int)((pix / W) % H);
  const int n = (int)(pix / ((long long)W * H));
  const long long base = (((long long)n * 2 * H + 2 * h) * 2 * W + 2 * w) * CV + cv;
  const uint4 a = dsrc[base], b = dsrc[base + CV], c = dsrc[base + (long long)2 * W * CV], d = dsrc[base + (long long)2 * W * CV + CV];
  uint4 o;
  o.x = add_bf16x2_f32(a.x, b.x, c.x, d.x); o.y = add_bf16x2_f32(a.y, b.y, c.y, d.y);
  o.z = add_bf16x2_f32(a.z, b.z, c.z, d.z); o.w = add_bf16x2_f32(a.w, b.w, c.w, d.w);
  ddst[idx] = o;
}

// parity planes: dst[(p*2+q)*N + n][h][w][:] = src[n][2h+p][2w+q][:]; to_planes=0 runs the inverse copy
__global__ void planes_kernel(const uint4* __restrict__ src, uint4* __restrict__ dst, int N, int H, int W, int CV, int to_planes) {
  const long long idx = gtid();  // index over the full-resolution tensor [N][H][W][CV]
  const long long total = (long long)N * H * W * CV;
  if (idx >= total) return;
  const int cv = (int)(idx % CV);
  const long long pix = idx / CV;
  const int w = (int)(pix % W);
  const int h = (int)((pix / W) % H);
  const int n = (int)(pix / ((long long)W * H));
  const int Ho = H / 2, Wo = W / 2;
  const long long pidx = ((((long long)((h & 1) * 2 + (w & 1)) * N + n) * Ho + (h >> 1)) * Wo + (w >> 1)) * CV + cv;
  if (to_planes) dst[pidx] = src[idx]; else dst[idx] = src[pidx];
}

__global__ void concat_kernel(const uint4* __restrict__ a, int CVa, const uint4* __restrict__ b, int CVb, uint4* __restrict__ dst, long long rows) {
  const long long idx = gtid();
  const int CV = CVa + CVb;
  if (idx >= rows * CV) return;
  const long long r = idx / CV;
  const int c = (int)(idx - r * CV);
  dst[idx] = (c < CVa) ? a[r * CVa + c] : b[r * CVb + (c - CVa)];
}
__global__ void split_kernel(const uint4* __restrict__ src, uint4* __restrict__ a, int CVa, uint4* __restrict__ b, int CVb, long long rows,
                             int accumulate_a) {
  const long long idx = gtid();
  const int CV = CVa + CVb;
  if (idx >= rows * CV) return;
  const long long r = idx / CV;
  const int c = (int)(idx - r * CV);
  const uint4 v = src[idx];
  if (c < CVa) {
    uint4* p = a + r * CVa + c;
    if (accumulate_a) {
      const uint4 o = *p;
      uint4 s;
      float2 x, y;
      x = unpack_bf16x2(o.x); y = unpack_bf16x2(v.x); s.x = pack_bf16x2(x.x + y.x, x.y + y.y);
      x = unpack_bf16x2(o.y); y = unpack_bf16x2(v.y); s.y = pack_bf16x2(x.x + y.x, x.y + y.y);
      x = unpack_bf16x2(o.z); y = unpack_bf16x2(v.z); s.z = pack_bf16x2(x.x + y.x, x.y + y.y);
      x = unpack_bf16x2(o.w); y = unpack_bf16x2(v.w); s.w = pack_bf16x2(x.x + y.x, x.y + y.y);
      *p = s;
    } else {
      *p = v;
    }
  } else if (b) {
    b[r * CVb + (c - CVa)] = v;
  }
}

// y = s0*a + s1*b (scales == NULL -> 1,1)
__global__ void axpby_kernel(const uint4* __restrict__ a, const uint4* __restrict__ b, const float* __restrict__ scales, uint4* __restrict__ y,
                             long long nvec) {
  const long long idx = gtid();
  if (idx >= nvec) return;
  const float s0 = scales ? scales[0] : 1.f, s1 = scales ? scales[1] : 1.f;
  const uint4 u = a[idx], v = b[idx];
  uint4 o;
  float2 x, z;
  x = unpack_bf16x2(u.x); z = unpack_bf16x2(v.x); o.x = pack_bf16x2(s0 * x.x + s1 * z.x, s0 * x.y + s1 * z.y);
  x = unpack_bf16x2(u.y); z = unpack_bf16x2(v.y); o.y = pack_bf16x2(s0 * x.x + s1 * z.x, s0 * x.y + s1 * z.y);
  x = unpack_bf16x2(u.z); z = unpack_bf16x2(v.z); o.z = pack_bf16x2(s0 * x.x + s1 * z.x, s0 * x.y + s1 * z.y);
  x = unpack_bf16x2(u.w); z = unpack_bf16x2(v.w); o.w = pack_bf16x2(s0 * x.x + s1 * z.x, s0 * x.y + s1 * z.y);
  y[idx] = o;
}

__global__ void silu_f32_kernel(const float* __restrict__ x, float* __restrict__ y, long long n) {
  const long long i = gtid();
  if (i < n) y[i] = silu_f(x[i]);
}

// column sums of a bf16 [rows][ldx] matrix: grid (blocks of 32 column vectors = 256 columns, row chunks); 256 threads =
// 32 column vectors (16 B each, 512 B contiguous per warp) x 8 row lanes, 4 loads in flight; fp32 atomics into out
__global__ void __launch_bounds__(256) colsum_kernel(const bf16* __restrict__ x, long long ldx, long long rows, int cols, long long rows_per_cta,
                                                     float* __restrict__ out) {
  __shared__ float sh[8][256 + 8];
  const int cvl = threadIdx.x & 31, rl = threadIdx.x >> 5;
  const int c0 = (blockIdx.x * 32 + cvl) * 8;
  const long long r0 = (long long)blockIdx.y * rows_per_cta;
  const long long r1 = min(r0 + rows_per_cta, rows);
  float a[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) a[k] = 0.f;
  if (c0 < cols) {
    long long r = r0 + rl;
    for (; r + 24 < r1; r += 32) {
      uint4 u[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) u[q] = *reinterpret_cast<const uint4*>(x + (r + 8 * q) * ldx + c0);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const uint32_t w[4] = {u[q].x, u[q].y, u[q].z, u[q].w};
#pragma unroll
        for (int k = 0; k < 4; ++k) { const float2 v = unpack_bf16x2(w[k]); a[2 * k] += v.x; a[2 * k + 1] += v.y; }
      }
    }
    for (; r < r1; r += 8) {
      const uint4 u = *reinterpret_cast<const uint4*>(x + r * ldx + c0);
      const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) { const float2 v = unpack_bf16x2(w[k]); a[2 * k] += v.x; a[2 * k + 1] += v.y; }
    }
  }
#pragma unroll
  for (int k = 0; k < 8; ++k) sh[rl][cvl * 8 + k] = a[k];
  __syncthreads();
  {
    const int c = threadIdx.x;  // 256 columns of this block
    float sacc = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) sacc += sh[k][c];
    const int cc = blockIdx.x * 256 + c;
    if (cc < cols) atomicAdd(out + cc, sacc);
  }
}

// GEGLU backward without a bias gradient: one thread per 8 columns of one row (maximum memory-level parallelism)
__global__ void geglu_bwd_plain_kernel(const bf16* __restrict__ pre, long long ldpre, const bf16* __restrict__ dout, long long lddo,
                                       bf16* __restrict__ dpre, long long lddpre, long long rows, int h) {
  const long long idx = gtid();
  const int hv = h / 8;
  if (idx >= rows * hv) return;
  const long long r = idx / hv;
  const int c = (int)(idx - r * hv) * 8;
  const uint4 uv = *reinterpret_cast<const uint4*>(pre + r * ldpre + c);
  const uint4 ug = *reinterpret_cast<const uint4*>(pre + r * ldpre + h + c);
  const uint4 ud = *reinterpret_cast<const uint4*>(dout + r * lddo + c);
  const uint32_t v[4] = {uv.x, uv.y, uv.z, uv.w}, g[4] = {ug.x, ug.y, ug.z, ug.w}, d[4] = {ud.x, ud.y, ud.z, ud.w};
  uint32_t ov[4], og[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const float2 fv = unpack_bf16x2(v[k]), fg = unpack_bf16x2(g[k]), fd = unpack_bf16x2(d[k]);
    ov[k] = pack_bf16x2(fd.x * gelu_erf_f(fg.x), fd.y * gelu_erf_f(fg.y));
    og[k] = pack_bf16x2(fd.x * fv.x * gelu_erf_grad_f(fg.x), fd.y * fv.y * gelu_erf_grad_f(fg.y));
  }
  *reinterpret_cast<uint4*>(dpre + r * lddpre + c) = make_uint4(ov[0], ov[1], ov[2], ov[3]);
  *reinterpret_cast<uint4*>(dpre + r * lddpre + h + c) = make_uint4(og[0], og[1], og[2], og[3]);
}

// GEGLU backward. pre = [value | gate] (bf16, the saved projection), dout [rows][h]:
//   dpre[:, :h] = dout * gelu(gate),  dpre[:, h:] = dout * value * gelu'(gate)
// and, fused, the bias gradient of the projection = column sums of the (bf16-rounded) dpre it writes — saving the separate
// column-sum pass over the [rows][2h] tensor (the largest activation gradient of a transformer block).
// Block = 32 column vectors (8 columns each) x 8 row lanes, rows streamed in chunks of rows_per_cta like colsum_kernel.
__global__ void __launch_bounds__(256, 2) geglu_bwd_kernel(const bf16* __restrict__ pre, long long ldpre, const bf16* __restrict__ dout, long long lddo,
                                                        bf16* __restrict__ dpre, long long lddpre, long long rows, int h, long long rows_per_cta,
                                                        float* __restrict__ bias_grad) {
  __shared__ float sh[8][2][256 + 8];
  const int cvl = threadIdx.x & 31, rl = threadIdx.x >> 5;
  const int c = (blockIdx.x * 32 + cvl) * 8;
  const long long r0 = (long long)blockIdx.y * rows_per_cta;
  const long long r1 = min(r0 + rows_per_cta, rows);
  float av[8], ag[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) { av[k] = 0.f; ag[k] = 0.f; }
  if (c < h) {
    for (long long r = r0 + rl; r < r1; r += 32) {
      // four rows in flight per thread (9 x 16-byte loads issued before any arithmetic)
      uint4 uv[4], ug[4], ud[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        if (r + 8 * q < r1) {
          uv[q] = *reinterpret_cast<const uint4*>(pre + (r + 8 * q) * ldpre + c);
          ug[q] = *reinterpret_cast<const uint4*>(pre + (r + 8 * q) * ldpre + h + c);
          ud[q] = *reinterpret_cast<const uint4*>(dout + (r + 8 * q) * lddo + c);
        }
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        if (r + 8 * q >= r1) break;
        const uint32_t v[4] = {uv[q].x, uv[q].y, uv[q].z, uv[q].w}, g[4] = {ug[q].x, ug[q].y, ug[q].z, ug[q].w}, d[4] = {ud[q].x, ud[q].y, ud[q].z, ud[q].w};
        uint32_t ov[4], og[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float2 fv = unpack_bf16x2(v[k]), fg = unpack_bf16x2(g[k]), fd = unpack_bf16x2(d[k]);
          ov[k] = pack_bf16x2(fd.x * gelu_erf_f(fg.x), fd.y * gelu_erf_f(fg.y));
          og[k] = pack_bf16x2(fd.x * fv.x * gelu_erf_grad_f(fg.x), fd.y * fv.y * gelu_erf_grad_f(fg.y));
          const float2 rv = unpack_bf16x2(ov[k]), rg = unpack_bf16x2(og[k]);
          av[2 * k] += rv.x; av[2 * k + 1] += rv.y;
          ag[2 * k] += rg.x; ag[2 * k + 1] += rg.y;
        }
        const long long rr = r + 8 * q;
        *reinterpret_cast<uint4*>(dpre + rr * lddpre + c) = make_uint4(ov[0], ov[1], ov[2], ov[3]);
        *reinterpret_cast<uint4*>(dpre + rr * lddpre + h + c) = make_uint4(og[0], og[1], og[2], og[3]);
      }
    }
  }
#pragma unroll
  for (int k = 0; k < 8; ++k) { sh[rl][0][cvl * 8 + k] = av[k]; sh[rl][1][cvl * 8 + k] = ag[k]; }
  __syncthreads();
  {
    const int cc = threadIdx.x;   // 256 columns of this block, both halves
    float s0 = 0.f, s1 = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) { s0 += sh[k][0][cc]; s1 += sh[k][1][cc]; }
    const int col = blockIdx.x * 256 + cc;
    if (col < h) { atomicAdd(bias_grad + col, s0); atomicAdd(bias_grad + h + col, s1); }
  }
}

__global__ void unprep_conv_grad_kernel(const float* __restrict__ src, float* __restrict__ dst, int O, int I, int taps, int i_pad) {
  const long long idx = gtid();  // over dst [O][I][taps]
  if (idx >= (long long)O * I * taps) return;
  const int t = (int)(idx % taps);
  const int i = (int)((idx / taps) % I);
  const int o = (int)(idx / ((long long)taps * I));
  dst[idx] += src[((long long)o * taps + t) * i_pad + i];
}

__global__ void __launch_bounds__(256) dot_diff_kernel(const uint4* __restrict__ dy, const uint4* __restrict__ a, const uint4* __restrict__ b,
                                                       long long nvec, float* out) {
  float acc = 0.f;
  for (long long i = gtid(); i < nvec; i += (long long)gridDim.x * blockDim.x) {
    const uint4 d = dy[i], x = a[i], y = b[i];
    const uint32_t dd[4] = {d.x, d.y, d.z, d.w}, xx[4] = {x.x, x.y, x.z, x.w}, yy[4] = {y.x, y.y, y.z, y.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float2 fd = unpack_bf16x2(dd[k]), fx = unpack_bf16x2(xx[k]), fy = unpack_bf16x2(yy[k]);
      acc += fd.x * (fx.x - fy.x) + fd.y * (fx.y - fy.y);
    }
  }
  acc = warp_sum(acc);
  __shared__ float sh[8];
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int k = 0; k < 8; ++k) s += sh[k];
    atomicAdd(out, s);
  }
}

__global__ void silu_bwd_f32_kernel(const float* __restrict__ x, const float* __restrict__ dy, float* __restrict__ dx, long long n) {
  const long long i = gtid();
  if (i < n) dx[i] = dy[i] * silu_grad_f(x[i]);
}

// epilogue of a split-K contraction: out = s0*act(ws + bias + rowbias[m/div]) + s1*res1 + s2*res2  (bf16), 8 columns per thread
__global__ void __launch_bounds__(256) splitk_epilogue_kernel(float* __restrict__ ws, long long ldw, bf16* __restrict__ out, long long ldo,
                                                              long long rows, int cols, const float* __restrict__ bias,
                                                              const float* __restrict__ rowbias, int rb_div, long long ldrb,
                                                              const bf16* __restrict__ res1, long long ldr1, const bf16* __restrict__ res2,
                                                              long long ldr2, const float* __restrict__ scales, int act) {
  const int cv = cols / 8;
  const long long idx = gtid();
  if (idx >= rows * cv) return;
  const long long r = idx / cv;
  const int c = (int)(idx - r * cv) * 8;
  float s0 = 1.f, s1 = 1.f, s2 = 1.f;
  if (scales) { s0 = scales[0]; s1 = scales[1]; s2 = scales[2]; }
  const float4 a = *reinterpret_cast<const float4*>(ws + r * ldw + c);
  const float4 b = *reinterpret_cast<const float4*>(ws + r * ldw + c + 4);
  // consume: leave the workspace zeroed for the next split-K accumulation
  *reinterpret_cast<float4*>(ws + r * ldw + c) = make_float4(0.f, 0.f, 0.f, 0.f);
  *reinterpret_cast<float4*>(ws + r * ldw + c + 4) = make_float4(0.f, 0.f, 0.f, 0.f);
  float f[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
  if (bias) {
#pragma unroll
    for (int k = 0; k < 8; ++k) f[k] += bias[c + k];
  }
  if (rowbias) {
    const float* rb = rowbias + (r / rb_div) * ldrb + c;
#pragma unroll
    for (int k = 0; k < 8; ++k) f[k] += rb[k];
  }
  if (act == SVDX_ACT_GELU) {
#pragma unroll
    for (int k = 0; k < 8; ++k) f[k] = gelu_erf_f(f[k]);
  }
#pragma unroll
  for (int k = 0; k < 8; ++k) f[k] *= s0;
  if (res1) {
    const uint4 u = *reinterpret_cast<const uint4*>(res1 + r * ldr1 + c);
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) { const float2 v = unpack_bf16x2(w[k]); f[2 * k] += s1 * v.x; f[2 * k + 1] += s1 * v.y; }
  }
  if (res2) {
    const uint4 u = *reinterpret_cast<const uint4*>(res2 + r * ldr2 + c);
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) { const float2 v = unpack_bf16x2(w[k]); f[2 * k] += s2 * v.x; f[2 * k + 1] += s2 * v.y; }
  }
  *reinterpret_cast<uint4*>(out + r * ldo + c) =
      make_uint4(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]), pack_bf16x2(f[4], f[5]), pack_bf16x2(f[6], f[7]));
}

__global__ void blend_scales_kernel(const float* mix, float* out) {
  const float a = 1.f / (1.f + __expf(-mix[0]));
  out[0] = 1.f - a; out[1] = a; out[2] = 1.f - a; out[3] = 0.f;
  out[4] = 1.f - a; out[5] = 1.f; out[6] = 0.f; out[7] = a * (1.f - a);
  out[8] = 1.f - a; out[9] = 0.f; out[10] = 0.f; out[11] = 0.f;     // accumulator-only triple for the gradient GEMMs
  out[12] = a; out[13] = 0.f; out[14] = 1.f - a; out[15] = 0.f;      // {s, 0} pairs for svdx_axpby_bf16 (scaled copies)
}

__global__ void adamw_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, long long n,
                             float lr, float b1, float b2, float eps, float wd, float bc1, float bc2, float gscale, bf16* __restrict__ shadow) {
  const long long i = gtid();
  if (i >= n) return;
  const float gi = g[i] * gscale;
  float pi = p[i] * (1.f - lr * wd);
  const float mi = b1 * m[i] + (1.f - b1) * gi;
  const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
  m[i] = mi;
  v[i] = vi;
  const float denom = sqrtf(vi) / sqrtf(bc2) + eps;
  pi -= (lr / bc1) * mi / denom;
  p[i] = pi;
  if (shadow) shadow[i] = __float2bfloat16(pi);   // bf16 operand copy of the updated weight, same flat offset
}

// CUDA-graph-safe form: every scalar that changes between steps lives in a small device buffer
//   state[0] lr  [1] beta1  [2] beta2  [3] eps  [4] weight_decay  [5] step (float, exact up to 2^24)  [6] 1-beta1^step  [7] 1-beta2^step
// adamw_tick advances the step count and the bias corrections on the device, so a captured graph that contains
// tick + update replays torch.optim.AdamW's step sequence; the learning rate is whatever the host last wrote to state[0].
__global__ void adamw_tick_kernel(float* state) {
  const float step = state[5] + 1.f;
  state[5] = step;
  state[6] = 1.f - powf(state[1], step);
  state[7] = 1.f - powf(state[2], step);
}
__global__ void adamw_state_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, long long n4,
                                   long long n, const float* __restrict__ state, float gscale, bf16* __restrict__ shadow) {
  const long long i4 = gtid();
  if (i4 >= n4) return;
  const float lr = state[0], b1 = state[1], b2 = state[2], eps = state[3], wd = state[4], bc1 = state[6], bc2 = state[7];
  const float decay = 1.f - lr * wd, step_size = lr / bc1, inv_sqrt_bc2 = rsqrtf(bc2);
  const long long i = i4 * 4;
  if (i + 3 < n) {
    const float4 g4 = *reinterpret_cast<const float4*>(g + i);
    float4 p4 = *reinterpret_cast<float4*>(p + i), m4 = *reinterpret_cast<float4*>(m + i), v4 = *reinterpret_cast<float4*>(v + i);
    float pp[4] = {p4.x, p4.y, p4.z, p4.w}, mm[4] = {m4.x, m4.y, m4.z, m4.w}, vv[4] = {v4.x, v4.y, v4.z, v4.w};
    const float gg[4] = {g4.x * gscale, g4.y * gscale, g4.z * gscale, g4.w * gscale};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      mm[k] = b1 * mm[k] + (1.f - b1) * gg[k];
      vv[k] = b2 * vv[k] + (1.f - b2) * gg[k] * gg[k];
      pp[k] = pp[k] * decay - step_size * mm[k] / (sqrtf(vv[k]) * inv_sqrt_bc2 + eps);
    }
    *reinterpret_cast<float4*>(p + i) = make_float4(pp[0], pp[1], pp[2], pp[3]);
    *reinterpret_cast<float4*>(m + i) = make_float4(mm[0], mm[1], mm[2], mm[3]);
    *reinterpret_cast<float4*>(v + i) = make_float4(vv[0], vv[1], vv[2], vv[3]);
    if (shadow) {
      uint2 o;
      o.x = pack_bf16x2(pp[0], pp[1]);
      o.y = pack_bf16x2(pp[2], pp[3]);
      *reinterpret_cast<uint2*>(shadow + i) = o;
    }
  } else {
    for (long long k = i; k < n; ++k) {
      const float gi = g[k] * gscale;
      const float mi = b1 * m[k] + (1.f - b1) * gi, vi = b2 * v[k] + (1.f - b2) * gi * gi;
      const float pi = p[k] * decay - step_size * mi / (sqrtf(vi) * inv_sqrt_bc2 + eps);
      m[k] = mi; v[k] = vi; p[k] = pi;
      if (shadow) shadow[k] = __float2bfloat16(pi);
    }
  }
}

// Data-parallel optimizer step as ONE kernel over NVLink peer memory: reduce-scatter + AdamW + all-gather fused.
// Rank r owns the arena slice [lo, lo + n). For every 4 owned elements it LOADS that slice of every rank's fp32 gradient
// arena (world - 1 of them through NVLink / NVSwitch peer mappings), sums in rank order (the same order on every rank: the
// owner is the only one that computes an element), applies AdamW (grad_scale = 1 / world -> the mean gradient) to its fp32
// master / moments, and STORES the bf16 operand value into every rank's shadow arena. Versus NCCL reduce-scatter -> AdamW ->
// all-gather: the same NVLink bytes, but no intermediate pass over HBM (the summed gradient and the local shadow slice are
// never written and re-read), one launch, and the link transfer overlaps the optimizer arithmetic load by load.
// The callers order it between two cross-rank barriers (all gradients final before / all shadows complete after).
struct AdamP2P {
  const float* grad[16];
  bf16* shadow[16];
};
__global__ void __launch_bounds__(256) adamw_p2p_kernel(float* __restrict__ p, float* __restrict__ m, float* __restrict__ v, const __grid_constant__ AdamP2P ptr,
                                                        int world, long long lo, long long n4, const float* __restrict__ state, float gscale) {
  const float lr = state[0], b1 = state[1], b2 = state[2], eps = state[3], wd = state[4], bc1 = state[6], bc2 = state[7];
  const float decay = 1.f - lr * wd, step_size = lr / bc1, inv_sqrt_bc2 = rsqrtf(bc2);
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long i4 = gtid(); i4 < n4; i4 += stride) {
    const long long i = i4 * 4;
    float4 g4 = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 1
    for (int r0 = 0; r0 < world; r0 += 4) {
      // up to four ranks' loads in flight together (NVLink round trips are microseconds)
      float4 t[4];
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (r0 + k < world) t[k] = __ldcg(reinterpret_cast<const float4*>(ptr.grad[r0 + k] + lo + i));
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (r0 + k < world) { g4.x += t[k].x; g4.y += t[k].y; g4.z += t[k].z; g4.w += t[k].w; }
    }
    float4 p4 = *reinterpret_cast<float4*>(p + i), m4 = *reinterpret_cast<float4*>(m + i), v4 = *reinterpret_cast<float4*>(v + i);
    float pp[4] = {p4.x, p4.y, p4.z, p4.w}, mm[4] = {m4.x, m4.y, m4.z, m4.w}, vv[4] = {v4.x, v4.y, v4.z, v4.w};
    const float gg[4] = {g4.x * gscale, g4.y * gscale, g4.z * gscale, g4.w * gscale};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      mm[k] = b1 * mm[k] + (1.f - b1) * gg[k];
      vv[k] = b2 * vv[k] + (1.f - b2) * gg[k] * gg[k];
      pp[k] = pp[k] * decay - step_size * mm[k] / (sqrtf(vv[k]) * inv_sqrt_bc2 + eps);
    }
    *reinterpret_cast<float4*>(p + i) = make_float4(pp[0], pp[1], pp[2], pp[3]);
    *reinterpret_cast<float4*>(m + i) = make_float4(mm[0], mm[1], mm[2], mm[3]);
    *reinterpret_cast<float4*>(v + i) = make_float4(vv[0], vv[1], vv[2], vv[3]);
    uint2 o;
    o.x = pack_bf16x2(pp[0], pp[1]);
    o.y = pack_bf16x2(pp[2], pp[3]);
    for (int r = 0; r < world; ++r) *reinterpret_cast<uint2*>(ptr.shadow[r] + lo + i) = o;
  }
  __threadfence_system();     // the peer stores are performed system-wide before this kernel counts as complete
}

// row softmax of a bf16 score matrix, y[r][:] = softmax(scale * x[r][:]) (fp32 arithmetic, in place allowed): the single-head,
// head_dim 512 attention of the VAE encoder's mid block goes through two GEMMs and this kernel (its S x S scores are small).
// One CTA per row; a row of <= 16 K columns stays L1/L2 resident over the three passes.
__global__ void __launch_bounds__(256) softmax_rows_kernel(const bf16* __restrict__ x, long long ldx, int cols, float scale, bf16* __restrict__ y,
                                                           long long ldy) {
  __shared__ float sh[8];
  const bf16* xr = x + (long long)blockIdx.x * ldx;
  bf16* yr = y + (long long)blockIdx.x * ldy;
  const int nv = cols / 8;
  const float sc = scale * 1.4426950408889634f;
  float m = -INFINITY;
  for (int v = threadIdx.x; v < nv; v += blockDim.x) {
    const uint4 u = *reinterpret_cast<const uint4*>(xr + v * 8);
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) { const float2 a = unpack_bf16x2(w[k]); m = fmaxf(m, fmaxf(a.x, a.y)); }
  }
  m = warp_max(m);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = m;
  __syncthreads();
  m = sh[0];
#pragma unroll
  for (int k = 1; k < 8; ++k) m = fmaxf(m, sh[k]);
  __syncthreads();
  const float msc = m * sc;
  float l = 0.f;
  for (int v = threadIdx.x; v < nv; v += blockDim.x) {
    const uint4 u = *reinterpret_cast<const uint4*>(xr + v * 8);
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) { const float2 a = unpack_bf16x2(w[k]); l += exp2_fast(fmaf(a.x, sc, -msc)) + exp2_fast(fmaf(a.y, sc, -msc)); }
  }
  l = warp_sum(l);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = l;
  __syncthreads();
  l = 0.f;
#pragma unroll
  for (int k = 0; k < 8; ++k) l += sh[k];
  const float inv = 1.0f / l;
  for (int v = threadIdx.x; v < nv; v += blockDim.x) {
    const uint4 u = *reinterpret_cast<const uint4*>(xr + v * 8);
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
    uint32_t o[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float2 a = unpack_bf16x2(w[k]);
      o[k] = pack_bf16x2(exp2_fast(fmaf(a.x, sc, -msc)) * inv, exp2_fast(fmaf(a.y, sc, -msc)) * inv);
    }
    *reinterpret_cast<uint4*>(yr + v * 8) = make_uint4(o[0], o[1], o[2], o[3]);
  }
}

// ---- skinny products of the [B, C] conditioning vectors (time-embedding MLPs, all 44 time_emb_proj at once, the 1-key image
// cross-attention collapse to_out(to_v(e)), their gradients): M = B rows. A 128-row tensor-core tile would be > 99 % padding and the
// launch is latency-bound (17 us for a 1 x 1280 x 1280 product on the tcgen05 kernel); these are weight-streaming GEMVs.
// out[m][n] = sum_k a[m][k] * w[n][k] (+ bias[n]), m < MR <= 8: one warp per output column, lanes stride K in 16-byte vectors.
template <int MR>
__global__ void __launch_bounds__(256) gemv_kernel(const bf16* __restrict__ a, long long lda, const bf16* __restrict__ w, long long ldw, int M, int N,
                                                   int K, const float* __restrict__ bias, void* __restrict__ out, long long ldo, int out_f32,
                                                   float scale, int accumulate) {
  const long long n = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (n >= N) return;
  float acc[MR];
#pragma unroll
  for (int m = 0; m < MR; ++m) acc[m] = 0.f;
  const bf16* wr = w + n * ldw;
  for (int v = lane; v < K / 8; v += 32) {
    const uint4 uw = __ldg(reinterpret_cast<const uint4*>(wr + v * 8));
    const uint32_t ww[4] = {uw.x, uw.y, uw.z, uw.w};
#pragma unroll
    for (int m = 0; m < MR; ++m) {
      if (m < M) {
        const uint4 ua = __ldg(reinterpret_cast<const uint4*>(a + m * lda + v * 8));
        const uint32_t aa[4] = {ua.x, ua.y, ua.z, ua.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float2 x = unpack_bf16x2(aa[k]), y = unpack_bf16x2(ww[k]);
          acc[m] = fmaf(x.x, y.x, acc[m]);
          acc[m] = fmaf(x.y, y.y, acc[m]);
        }
      }
    }
  }
#pragma unroll
  for (int m = 0; m < MR; ++m) acc[m] = warp_sum(acc[m]);
  if (lane == 0) {
    const float b = bias ? bias[n] : 0.f;
#pragma unroll
    for (int m = 0; m < MR; ++m) {
      if (m < M) {
        float r = fmaf(scale, acc[m], b);
        if (out_f32) {
          float* o = reinterpret_cast<float*>(out) + m * ldo + n;
          *o = accumulate ? *o + r : r;
        } else {
          bf16* o = reinterpret_cast<bf16*>(out) + m * ldo + n;
          *o = __float2bfloat16(accumulate ? __bfloat162float(*o) + r : r);
        }
      }
    }
  }
}

// g[o][k] += s * sum_{t < T} dy[t][o] * x[t][k]   (T <= 8 token rows: the weight gradient of a skinny product), 4 columns per thread
__global__ void outer_accum_kernel(const bf16* __restrict__ dy, long long lddy, const bf16* __restrict__ x, long long ldx, int T, int O, int K,
                                   const float* __restrict__ scale, float* __restrict__ g, long long ldg) {
  const long long idx = gtid();
  const int kv = K / 4;
  if (idx >= (long long)O * kv) return;
  const int o = (int)(idx / kv);
  const int k = (int)(idx - (long long)o * kv) * 4;
  const float s = scale ? scale[0] : 1.f;
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
  for (int t = 0; t < T; ++t) {
    const float d = __bfloat162float(dy[t * lddy + o]);
    const uint2 u = *reinterpret_cast<const uint2*>(x + t * ldx + k);
    const float2 p = unpack_bf16x2(u.x), q = unpack_bf16x2(u.y);
    a0 = fmaf(d, p.x, a0); a1 = fmaf(d, p.y, a1); a2 = fmaf(d, q.x, a2); a3 = fmaf(d, q.y, a3);
  }
  float4* gp = reinterpret_cast<float4*>(g + (long long)o * ldg + k);
  float4 cur = *gp;
  cur.x = fmaf(s, a0, cur.x); cur.y = fmaf(s, a1, cur.y); cur.z = fmaf(s, a2, cur.z); cur.w = fmaf(s, a3, cur.w);
  *gp = cur;
}

struct TransposeJob {
  long long src_off;   // element offset into the bf16 source arena
  bf16* dst;           // [I][O] destination
  int O, I;
};

// many 2-D transposes dst[i][o] = src[o][i] (bf16) in ONE launch: block -> (job, 64x64 tile) through a tile prefix
// table; 4-byte (bf16x2) global accesses so that a warp row covers a full 128-byte line on both sides.
constexpr int TR_TILE = 64;
__global__ void multi_transpose_kernel(const bf16* __restrict__ src_base, const TransposeJob* __restrict__ jobs,
                                       const int* __restrict__ tile_prefix, int njobs) {
  __shared__ bf16 tile[TR_TILE][TR_TILE + 2];
  int lo = 0, hi = njobs - 1;
  const int b = blockIdx.x;
  while (lo < hi) {            // last job whose first tile <= b
    const int mid = (lo + hi + 1) >> 1;
    if (tile_prefix[mid] <= b) lo = mid; else hi = mid - 1;
  }
  const TransposeJob j = jobs[lo];
  const int t = b - tile_prefix[lo];
  const int tiles_x = (j.I + TR_TILE - 1) / TR_TILE;
  const int i0 = (t % tiles_x) * TR_TILE, o0 = (t / tiles_x) * TR_TILE;
  const bf16* src = src_base + j.src_off;
  const int tx = threadIdx.x, ty = threadIdx.y;
  const bool vec_in = (j.I % 2 == 0) && ((reinterpret_cast<uintptr_t>(src) & 3) == 0);
  const bool vec_out = (j.O % 2 == 0) && ((reinterpret_cast<uintptr_t>(j.dst) & 3) == 0);
  for (int r = ty; r < TR_TILE; r += blockDim.y) {
    const int o = o0 + r, i = i0 + 2 * tx;
    if (o < j.O) {
      if (vec_in && i + 1 < j.I) {
        const __nv_bfloat162 v = *reinterpret_cast<const __nv_bfloat162*>(src + (long long)o * j.I + i);
        tile[r][2 * tx] = v.x; tile[r][2 * tx + 1] = v.y;
      } else {
        if (i < j.I) tile[r][2 * tx] = src[(long long)o * j.I + i];
        if (i + 1 < j.I) tile[r][2 * tx + 1] = src[(long long)o * j.I + i + 1];
      }
    }
  }
  __syncthreads();
  for (int r = ty; r < TR_TILE; r += blockDim.y) {
    const int i = i0 + r, o = o0 + 2 * tx;
    if (i < j.I) {
      if (vec_out && o + 1 < j.O) {
        __nv_bfloat162 v;
        v.x = tile[2 * tx][r]; v.y = tile[2 * tx + 1][r];
        *reinterpret_cast<__nv_bfloat162*>(j.dst + (long long)i * j.O + o) = v;
      } else {
        if (o < j.O) j.dst[(long long)i * j.O + o] = tile[2 * tx][r];
        if (o + 1 < j.O) j.dst[(long long)i * j.O + o + 1] = tile[2 * tx + 1][r];
      }
    }
  }
}

}  // namespace svdx

using namespace svdx;
#define ST(s) reinterpret_cast<cudaStream_t>(s)

extern "C" int svdx_prep_weight(const void* src, int32_t src_bf16, void* dst, int32_t mode, int32_t O, int32_t I, int32_t taps,
                                int32_t i_pad, void* stream) {
  if (!src || !dst || O <= 0 || I <= 0 || taps <= 0 || mode < 0 || mode > 3 || src_bf16 < 0 || src_bf16 > 2)
    return svdx_fail(SVDX_E_BADARG, "prep_weight: bad arguments (source dtype code: 0 fp32, 1 bf16, 2 fp16)");
  if ((mode == 0 || mode == 1) && taps != 1) return svdx_fail(SVDX_E_BADARG, "prep_weight: modes 0/1 need taps == 1");
  if (mode == 2 && i_pad < I) return svdx_fail(SVDX_E_BADARG, "prep_weight: i_pad < I");
  bf16* d = reinterpret_cast<bf16*>(dst);
  if (mode == 1) {
    dim3 grid((I + 31) / 32, (O + 31) / 32), block(32, 8);
    if (src_bf16 == 1) prep_transpose_kernel<bf16><<<grid, block, 0, ST(stream)>>>(reinterpret_cast<const bf16*>(src), d, O, I);
    else if (src_bf16 == 2) prep_transpose_kernel<__half><<<grid, block, 0, ST(stream)>>>(reinterpret_cast<const __half*>(src), d, O, I);
    else prep_transpose_kernel<float><<<grid, block, 0, ST(stream)>>>(reinterpret_cast<const float*>(src), d, O, I);
  } else {
    const long long total = mode == 0 ? (long long)O * I : mode == 2 ? (long long)O * taps * i_pad : (long long)I * taps * O;
    if (src_bf16 == 1) prep_gather_kernel<bf16><<<nblocks(total), 256, 0, ST(stream)>>>(reinterpret_cast<const bf16*>(src), d, mode, O, I, taps, i_pad);
    else if (src_bf16 == 2) prep_gather_kernel<__half><<<nblocks(total), 256, 0, ST(stream)>>>(reinterpret_cast<const __half*>(src), d, mode, O, I, taps, i_pad);
    else prep_gather_kernel<float><<<nblocks(total), 256, 0, ST(stream)>>>(reinterpret_cast<const float*>(src), d, mode, O, I, taps, i_pad);
  }
  SVDX_CHECK_LAUNCH("prep_weight");
  return SVDX_OK;
}

extern "C" int svdx_cast_f32_bf16(const float* src, void* dst, int64_t n, void* stream) {
  if (!src || !dst || n <= 0 || (reinterpret_cast<uintptr_t>(src) & 15) || (reinterpret_cast<uintptr_t>(dst) & 7))
    return svdx_fail(SVDX_E_BADARG, "cast_f32_bf16: bad arguments");
  cast_f32_bf16_kernel<<<nblocks((n + 3) / 4), 256, 0, ST(stream)>>>(src, reinterpret_cast<bf16*>(dst), n);
  SVDX_CHECK_LAUNCH("cast_f32_bf16");
  return SVDX_OK;
}
extern "C" int svdx_cast_bf16_f32(const void* src, float* dst, int64_t n, void* stream) {
  if (!src || !dst || n <= 0) return svdx_fail(SVDX_E_BADARG, "cast_bf16_f32: bad arguments");
  cast_bf16_f32_kernel<<<nblocks(n), 256, 0, ST(stream)>>>(reinterpret_cast<const bf16*>(src), dst, n);
  SVDX_CHECK_LAUNCH("cast_bf16_f32");
  return SVDX_OK;
}

extern "C" int svdx_cast_f16_f32(const void* src, float* dst, int64_t n, void* stream) {
  if (!src || !dst || n <= 0) return svdx_fail(SVDX_E_BADARG, "cast_f16_f32: bad arguments");
  cast_f16_f32_kernel<<<nblocks(n), 256, 0, ST(stream)>>>(reinterpret_cast<const __half*>(src), dst, n);
  SVDX_CHECK_LAUNCH("cast_f16_f32");
  return SVDX_OK;
}

extern "C" int svdx_nchw_to_nhwc(const void* src, int32_t src_bf16, void* dst, int32_t N, int32_t C, int32_t H, int32_t W, int32_t c_pad,
                                 void* stream) {
  if (!src || !dst || N <= 0 || C <= 0 || H <= 0 || W <= 0 || c_pad < C) return svdx_fail(SVDX_E_BADARG, "nchw_to_nhwc: bad arguments");
  const long long total = (long long)N * H * W * c_pad;
  if (src_bf16 == 1) nchw_to_nhwc_kernel<bf16><<<nblocks(total), 256, 0, ST(stream)>>>(reinterpret_cast<const bf16*>(src), reinterpret_cast<bf16*>(dst), N, C, H, W, c_pad);
  else if (src_bf16 == 2) nchw_to_nhwc_kernel<__half><<<nblocks(total), 256, 0, ST(stream)>>>(reinterpret_cast<const __half*>(src), reinterpret_cast<bf16*>(dst), N, C, H, W, c_pad);
  else nchw_to_nhwc_kernel<float><<<nblocks(total), 256, 0, ST(stream)>>>(reinterpret_cast<const float*>(src), reinterpret_cast<bf16*>(dst), N, C, H, W, c_pad);
  SVDX_CHECK_LAUNCH("nchw_to_nhwc");
  return SVDX_OK;
}
extern "C" int svdx_nhwc_to_nchw(const void* src, int64_t lds, void* dst, int32_t dst_bf16, int32_t N, int32_t C, int32_t H, int32_t W,
                                 void* stream) {
  if (!src || !dst || N <= 0 || C <= 0 || H <= 0 || W <= 0 || lds < C) return svdx_fail(SVDX_E_BADARG, "nhwc_to_nchw: bad arguments");
  const long long total = (long long)N * C * H * W;
  if (dst_bf16 == 1) nhwc_to_nchw_kernel<bf16><<<nblocks(total), 256, 0, ST(stream)>>>(reinterpret_cast<const bf16*>(src), lds, reinterpret_cast<bf16*>(dst), N, C, H, W);
  else if (dst_bf16 == 2) nhwc_to_nchw_kernel<__half><<<nblocks(total), 256, 0, ST(stream)>>>(reinterpret_cast<const bf16*>(src), lds, reinterpret_cast<__half*>(dst), N, C, H, W);
  else nhwc_to_nchw_kernel<float><<<nblocks(total), 256, 0, ST(stream)>>>(reinterpret_cast<const bf16*>(src), lds, reinterpret_cast<float*>(dst), N, C, H, W);
  SVDX_CHECK_LAUNCH("nhwc_to_nchw");
  return SVDX_OK;
}

static int vec_ok(const void* a, const void* b, int C) {
  return a && b && C > 0 && C % 8 == 0 && !(reinterpret_cast<uintptr_t>(a) & 15) && !(reinterpret_cast<uintptr_t>(b) & 15);
}

extern "C" int svdx_upsample2x(const void* src, void* dst, int32_t N, int32_t H, int32_t W, int32_t C, void* stream) {
  if (!vec_ok(src, dst, C) || N <= 0 || H <= 0 || W <= 0) return svdx_fail(SVDX_E_BADARG, "upsample2x: bad arguments");
  const long long total = (long long)N * 4 * H * W * (C / 8);
  upsample2x_kernel<<<nblocks(total), 256, 0, ST(stream)>>>(reinterpret_cast<const uint4*>(src), reinterpret_cast<uint4*>(dst), N, H, W, C / 8);
  SVDX_CHECK_LAUNCH("upsample2x");
  return SVDX_OK;
}
extern "C" int svdx_upsample2x_bwd(const void* dsrc, void* ddst, int32_t N, int32_t H, int32_t W, int32_t C, void* stream) {
  if (!vec_ok(dsrc, ddst, C) || N <= 0 || H <= 0 || W <= 0) return svdx_fail(SVDX_E_BADARG, "upsample2x_bwd: bad arguments");
  const long long total = (long long)N * H * W * (C / 8);
  upsample2x_bwd_kernel<<<nblocks(total), 256, 0, ST(stream)>>>(reinterpret_cast<const uint4*>(dsrc), reinterpret_cast<uint4*>(ddst), N, H, W, C / 8);
  SVDX_CHECK_LAUNCH("upsample2x_bwd");
  return SVDX_OK;
}
extern "C" int svdx_space_to_planes(const void* src, void* dst, int32_t N, int32_t H, int32_t W, int32_t C, void* stream) {
  if (!vec_ok(src, dst, C) || N <= 0 || H <= 0 || W <= 0 || H % 2 || W % 2) return svdx_fail(SVDX_E_BADARG, "space_to_planes: bad arguments");
  const long long total = (long long)N * H * W * (C / 8);
  planes_kernel<<<nblocks(total), 256, 0, ST(stream)>>>(reinterpret_cast<const uint4*>(src), reinterpret_cast<uint4*>(dst), N, H, W, C / 8, 1);
  SVDX_CHECK_LAUNCH("space_to_planes");
  return SVDX_OK;
}
extern "C" int svdx_planes_to_space(const void* src, void* dst, int32_t N, int32_t H, int32_t W, int32_t C, void* stream) {
  if (!vec_ok(src, dst, C) || N <= 0 || H <= 0 || W <= 0 || H % 2 || W % 2) return svdx_fail(SVDX_E_BADARG, "planes_to_space: bad arguments");
  const long long total = (long long)N * H * W * (C / 8);
  planes_kernel<<<nblocks(total), 256, 0, ST(stream)>>>(reinterpret_cast<const uint4*>(src), reinterpret_cast<uint4*>(dst), N, H, W, C / 8, 0);
  SVDX_CHECK_LAUNCH("planes_to_space");
  return SVDX_OK;
}

extern "C" int svdx_concat_channels(const void* a, int32_t Ca, const void* b, int32_t Cb, void* dst, int64_t rows, void* stream) {
  if (!vec_ok(a, dst, Ca) || !vec_ok(b, dst, Cb) || rows <= 0) return svdx_fail(SVDX_E_BADARG, "concat_channels: bad arguments");
  const long long total = rows * ((Ca + Cb) / 8);
  concat_kernel<<<nblocks(total), 256, 0, ST(stream)>>>(reinterpret_cast<const uint4*>(a), Ca / 8, reinterpret_cast<const uint4*>(b), Cb / 8,
                                                        reinterpret_cast<uint4*>(dst), rows);
  SVDX_CHECK_LAUNCH("concat_channels");
  return SVDX_OK;
}
extern "C" int svdx_split_channels(const void* src, void* a, int32_t Ca, void* b, int32_t Cb, int64_t rows, int32_t accumulate_a, void* stream) {
  if (!vec_ok(src, a, Ca) || Cb <= 0 || Cb % 8 || rows <= 0 || (b && (reinterpret_cast<uintptr_t>(b) & 15)))
    return svdx_fail(SVDX_E_BADARG, "split_channels: bad arguments");
  const long long total = rows * ((Ca + Cb) / 8);
  split_kernel<<<nblocks(total), 256, 0, ST(stream)>>>(reinterpret_cast<const uint4*>(src), reinterpret_cast<uint4*>(a), Ca / 8,
                                                       reinterpret_cast<uint4*>(b), Cb / 8, rows, accumulate_a);
  SVDX_CHECK_LAUNCH("split_channels");
  return SVDX_OK;
}

extern "C" int svdx_axpby_bf16(const void* a, const void* b, const float* scales, void* y, int64_t n, void* stream) {
  if (!a || !b || !y || n <= 0 || n % 8 || (reinterpret_cast<uintptr_t>(a) & 15) || (reinterpret_cast<uintptr_t>(b) & 15) ||
      (reinterpret_cast<uintptr_t>(y) & 15))
    return svdx_fail(SVDX_E_BADARG, "axpby_bf16: bad arguments (n %% 8, 16 B alignment)");
  axpby_kernel<<<nblocks(n / 8), 256, 0, ST(stream)>>>(reinterpret_cast<const uint4*>(a), reinterpret_cast<const uint4*>(b), scales,
                                                       reinterpret_cast<uint4*>(y), n / 8);
  SVDX_CHECK_LAUNCH("axpby_bf16");
  return SVDX_OK;
}
extern "C" int svdx_add_bf16(const void* a, const void* b, void* y, int64_t n, void* stream) { return svdx_axpby_bf16(a, b, nullptr, y, n, stream); }

extern "C" int svdx_silu_f32(const float* x, float* y, int64_t n, void* stream) {
  if (!x || !y || n <= 0) return svdx_fail(SVDX_E_BADARG, "silu_f32: bad arguments");
  silu_f32_kernel<<<nblocks(n), 256, 0, ST(stream)>>>(x, y, n);
  SVDX_CHECK_LAUNCH("silu_f32");
  return SVDX_OK;
}

extern "C" int svdx_colsum(const void* x, int64_t ldx, int64_t rows, int32_t cols, float* out, int32_t accumulate, void* stream) {
  if (!x || !out || rows <= 0 || cols <= 0 || cols % 8 || ldx % 8 || (reinterpret_cast<uintptr_t>(x) & 15))
    return svdx_fail(SVDX_E_BADARG, "colsum: bad arguments (cols, ldx multiples of 8; 16 B aligned)");
  if (!accumulate) cudaMemsetAsync(out, 0, sizeof(float) * cols, ST(stream));
  const int col_blocks = (cols + 255) / 256;
  long long chunks = (4LL * svdx_num_sms() + col_blocks - 1) / col_blocks;
  if (chunks < 1) chunks = 1;
  long long rows_per_cta = (rows + chunks - 1) / chunks;
  if (rows_per_cta < 64) rows_per_cta = 64;
  chunks = (rows + rows_per_cta - 1) / rows_per_cta;
  colsum_kernel<<<dim3(col_blocks, (unsigned)chunks), 256, 0, ST(stream)>>>(reinterpret_cast<const bf16*>(x), ldx, rows, cols, rows_per_cta, out);
  SVDX_CHECK_LAUNCH("colsum");
  return SVDX_OK;
}

extern "C" int svdx_geglu_bwd(const void* pre, int64_t ldpre, const void* dout, int64_t lddo, void* dpre, int64_t lddpre, int64_t rows,
                              int32_t h, float* bias_grad, void* stream) {
  if (!pre || !dout || !dpre || rows <= 0 || h <= 0 || h % 8 || ldpre % 8 || lddo % 8 || lddpre % 8)
    return svdx_fail(SVDX_E_BADARG, "geglu_bwd: bad arguments");
  if (!bias_grad) {
    geglu_bwd_plain_kernel<<<nblocks(rows * (h / 8)), 256, 0, ST(stream)>>>(reinterpret_cast<const bf16*>(pre), ldpre, reinterpret_cast<const bf16*>(dout), lddo,
                                                                      reinterpret_cast<bf16*>(dpre), lddpre, rows, h);
    SVDX_CHECK_LAUNCH("geglu_bwd");
    return SVDX_OK;
  }
  const int col_blocks = (h + 255) / 256;
  long long chunks = (16LL * svdx_num_sms() + col_blocks - 1) / col_blocks;
  if (chunks < 1) chunks = 1;
  long long rows_per_cta = (rows + chunks - 1) / chunks;
  rows_per_cta = (rows_per_cta + 31) / 32 * 32;
  if (rows_per_cta < 32) rows_per_cta = 32;
  chunks = (rows + rows_per_cta - 1) / rows_per_cta;
  geglu_bwd_kernel<<<dim3(col_blocks, (unsigned)chunks), 256, 0, ST(stream)>>>(reinterpret_cast<const bf16*>(pre), ldpre, reinterpret_cast<const bf16*>(dout),
                                                                             lddo, reinterpret_cast<bf16*>(dpre), lddpre, rows, h, rows_per_cta, bias_grad);
  SVDX_CHECK_LAUNCH("geglu_bwd");
  return SVDX_OK;
}

extern "C" int svdx_softmax_rows(const void* x, int64_t ldx, int64_t rows, int32_t cols, float scale, void* y, int64_t ldy, void* stream) {
  if (!x || !y || rows <= 0 || cols <= 0 || cols % 8 || ldx % 8 || ldy % 8 || (reinterpret_cast<uintptr_t>(x) & 15) || (reinterpret_cast<uintptr_t>(y) & 15) ||
      rows > 0x7fffffffLL)
    return svdx_fail(SVDX_E_BADARG, "softmax_rows: bad arguments (cols, ldx, ldy multiples of 8; 16 B aligned)");
  softmax_rows_kernel<<<(unsigned)rows, 256, 0, ST(stream)>>>(reinterpret_cast<const bf16*>(x), ldx, cols, scale, reinterpret_cast<bf16*>(y), ldy);
  SVDX_CHECK_LAUNCH("softmax_rows");
  return SVDX_OK;
}

extern "C" int svdx_gemv(const void* a, int64_t lda, const void* w, int64_t ldw, int32_t M, int32_t N, int32_t K, const float* bias, void* out,
                         int64_t ldo, int32_t out_dtype, float scale, int32_t accumulate, void* stream) {
  if (!a || !w || !out || M <= 0 || M > 8 || N <= 0 || K <= 0 || K % 8 || lda % 8 || ldw % 8 || (reinterpret_cast<uintptr_t>(a) & 15) ||
      (reinterpret_cast<uintptr_t>(w) & 15) || (out_dtype != SVDX_OUT_BF16 && out_dtype != SVDX_OUT_F32))
    return svdx_fail(SVDX_E_BADARG, "gemv: bad arguments (M <= 8, K, lda, ldw multiples of 8, 16 B aligned, bf16 / fp32 output)");
  const unsigned blocks = (unsigned)(((long long)N * 32 + 255) / 256);
  const int f32 = out_dtype == SVDX_OUT_F32;
  const bf16* ap = reinterpret_cast<const bf16*>(a);
  const bf16* wp = reinterpret_cast<const bf16*>(w);
  if (M == 1) gemv_kernel<1><<<blocks, 256, 0, ST(stream)>>>(ap, lda, wp, ldw, M, N, K, bias, out, ldo, f32, scale, accumulate);
  else if (M == 2) gemv_kernel<2><<<blocks, 256, 0, ST(stream)>>>(ap, lda, wp, ldw, M, N, K, bias, out, ldo, f32, scale, accumulate);
  else if (M <= 4) gemv_kernel<4><<<blocks, 256, 0, ST(stream)>>>(ap, lda, wp, ldw, M, N, K, bias, out, ldo, f32, scale, accumulate);
  else gemv_kernel<8><<<blocks, 256, 0, ST(stream)>>>(ap, lda, wp, ldw, M, N, K, bias, out, ldo, f32, scale, accumulate);
  SVDX_CHECK_LAUNCH("gemv");
  return SVDX_OK;
}

extern "C" int svdx_outer_accum(const void* dy, int64_t lddy, const void* x, int64_t ldx, int32_t T, int32_t O, int32_t K, const float* scale,
                                float* g, int64_t ldg, void* stream) {
  if (!dy || !x || !g || T <= 0 || T > 8 || O <= 0 || K <= 0 || K % 4 || ldx % 4 || ldg % 4 || (reinterpret_cast<uintptr_t>(x) & 7) ||
      (reinterpret_cast<uintptr_t>(g) & 15))
    return svdx_fail(SVDX_E_BADARG, "outer_accum: bad arguments (T <= 8, K, ldx, ldg multiples of 4, aligned)");
  outer_accum_kernel<<<nblocks((long long)O * (K / 4)), 256, 0, ST(stream)>>>(reinterpret_cast<const bf16*>(dy), lddy, reinterpret_cast<const bf16*>(x), ldx,
                                                                         T, O, K, scale, g, ldg);
  SVDX_CHECK_LAUNCH("outer_accum");
  return SVDX_OK;
}

extern "C" int svdx_blend_scales(const float* mix_factor, float* out3, void* stream) {
  if (!mix_factor || !out3) return svdx_fail(SVDX_E_BADARG, "blend_scales: null");
  blend_scales_kernel<<<1, 1, 0, ST(stream)>>>(mix_factor, out3);
  SVDX_CHECK_LAUNCH("blend_scales");
  return SVDX_OK;
}

extern "C" int svdx_adamw(float* p, const float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2, float eps,
                          float weight_decay, int32_t step, float grad_scale, void* shadow_bf16, void* stream) {
  if (!p || !g || !m || !v || n <= 0 || step < 1) return svdx_fail(SVDX_E_BADARG, "adamw: bad arguments");
  const float bc1 = 1.f - powf(beta1, (float)step), bc2 = 1.f - powf(beta2, (float)step);
  adamw_kernel<<<nblocks(n), 256, 0, ST(stream)>>>(p, g, m, v, n, lr, beta1, beta2, eps, weight_decay, bc1, bc2, grad_scale,
                                                   reinterpret_cast<bf16*>(shadow_bf16));
  SVDX_CHECK_LAUNCH("adamw");
  return SVDX_OK;
}

extern "C" int svdx_adamw_graph(float* p, const float* g, float* m, float* v, int64_t n, float* state, float grad_scale,
                                void* shadow_bf16, void* stream) {
  if (!p || !g || !m || !v || !state || n <= 0 || (reinterpret_cast<uintptr_t>(p) & 15) || (reinterpret_cast<uintptr_t>(g) & 15) ||
      (reinterpret_cast<uintptr_t>(m) & 15) || (reinterpret_cast<uintptr_t>(v) & 15) || (reinterpret_cast<uintptr_t>(shadow_bf16) & 7))
    return svdx_fail(SVDX_E_BADARG, "adamw_graph: bad arguments (16-byte aligned flat buffers, device state[8])");
  adamw_tick_kernel<<<1, 1, 0, ST(stream)>>>(state);
  const long long n4 = (n + 3) / 4;
  adamw_state_kernel<<<nblocks(n4), 256, 0, ST(stream)>>>(p, g, m, v, n4, n, state, grad_scale, reinterpret_cast<bf16*>(shadow_bf16));
  SVDX_CHECK_LAUNCH("adamw_graph");
  return SVDX_OK;
}

extern "C" int svdx_adamw_p2p(float* p, float* m, float* v, const void* const* grads, void* const* shadows, int32_t world, int64_t lo, int64_t n,
                              float* state, float grad_scale, int32_t tick, void* stream) {
  if (!p || !m || !v || !grads || !shadows || !state || world < 1 || world > 16 || n <= 0 || n % 4 || lo % 4 ||
      (reinterpret_cast<uintptr_t>(p) & 15) || (reinterpret_cast<uintptr_t>(m) & 15) || (reinterpret_cast<uintptr_t>(v) & 15))
    return svdx_fail(SVDX_E_BADARG, "adamw_p2p: bad arguments (world <= 16, slice offset / length multiples of 4, 16-byte aligned buffers)");
  AdamP2P ptr;
  for (int r = 0; r < 16; ++r) { ptr.grad[r] = nullptr; ptr.shadow[r] = nullptr; }
  for (int r = 0; r < world; ++r) {
    if (!grads[r] || !shadows[r] || (reinterpret_cast<uintptr_t>(grads[r]) & 15) || (reinterpret_cast<uintptr_t>(shadows[r]) & 7))
      return svdx_fail(SVDX_E_BADARG, "adamw_p2p: null / misaligned peer arena");
    ptr.grad[r] = reinterpret_cast<const float*>(grads[r]);
    ptr.shadow[r] = reinterpret_cast<bf16*>(shadows[r]);
  }
  if (tick) adamw_tick_kernel<<<1, 1, 0, ST(stream)>>>(state);
  const long long n4 = n / 4;
  // a few resident CTAs per SM, grid-stride: enough 16-byte loads in flight to cover the NVLink round trip
  long long blocks = (n4 + 255) / 256;
  const long long cap = (long long)svdx_num_sms() * 8;
  if (blocks > cap) blocks = cap;
  adamw_p2p_kernel<<<(unsigned)blocks, 256, 0, ST(stream)>>>(p, m, v, ptr, world, lo, n4, state, grad_scale);
  SVDX_CHECK_LAUNCH("adamw_p2p");
  return SVDX_OK;
}

extern "C" int svdx_multi_transpose(const void* src_base, const void* jobs, const int32_t* tile_prefix, int32_t njobs, int32_t total_tiles,
                                    void* stream) {
  if (!src_base || !jobs || !tile_prefix || njobs <= 0 || total_tiles <= 0) return svdx_fail(SVDX_E_BADARG, "multi_transpose: bad arguments");
  multi_transpose_kernel<<<total_tiles, dim3(32, 8), 0, ST(stream)>>>(reinterpret_cast<const bf16*>(src_base),
                                                                     reinterpret_cast<const TransposeJob*>(jobs), tile_prefix, njobs);
  SVDX_CHECK_LAUNCH("multi_transpose");
  return SVDX_OK;
}

extern "C" int svdx_unprep_conv_grad(const float* src, float* dst, int32_t O, int32_t I, int32_t taps, int32_t i_pad, void* stream) {
  if (!src || !dst || O <= 0 || I <= 0 || taps <= 0 || i_pad < I) return svdx_fail(SVDX_E_BADARG, "unprep_conv_grad: bad arguments");
  unprep_conv_grad_kernel<<<nblocks((long long)O * I * taps), 256, 0, ST(stream)>>>(src, dst, O, I, taps, i_pad);
  SVDX_CHECK_LAUNCH("unprep_conv_grad");
  return SVDX_OK;
}

extern "C" int svdx_dot_diff(const void* dy, const void* a, const void* b, int64_t n, float* out, void* stream) {
  if (!dy || !a || !b || !out || n <= 0 || n % 8) return svdx_fail(SVDX_E_BADARG, "dot_diff: bad arguments");
  long long nvec = n / 8;
  unsigned grid = nblocks(nvec);
  const unsigned cap = 4u * (unsigned)svdx_num_sms();
  if (grid > cap) grid = cap;
  dot_diff_kernel<<<grid, 256, 0, ST(stream)>>>(reinterpret_cast<const uint4*>(dy), reinterpret_cast<const uint4*>(a),
                                              reinterpret_cast<const uint4*>(b), nvec, out);
  SVDX_CHECK_LAUNCH("dot_diff");
  return SVDX_OK;
}

extern "C" int svdx_silu_bwd_f32(const float* x, const float* dy, float* dx, int64_t n, void* stream) {
  if (!x || !dy || !dx || n <= 0) return svdx_fail(SVDX_E_BADARG, "silu_bwd_f32: bad arguments");
  silu_bwd_f32_kernel<<<nblocks(n), 256, 0, ST(stream)>>>(x, dy, dx, n);
  SVDX_CHECK_LAUNCH("silu_bwd_f32");
  return SVDX_OK;
}

extern "C" int svdx_splitk_epilogue_act(float* ws, int64_t ldw, void* out, int64_t ldo, int64_t rows, int32_t cols, const float* bias,
                                        const float* rowbias, int32_t rowbias_div, int64_t ldrb, const void* res1, int64_t ldr1,
                                        const void* res2, int64_t ldr2, const float* scales, int32_t act, void* stream) {
  if (!ws || !out || rows <= 0 || cols <= 0 || cols % 8 || ldw % 4 || ldo % 8 || (res1 && ldr1 % 8) || (res2 && ldr2 % 8) ||
      (rowbias && rowbias_div <= 0) || (act != SVDX_ACT_NONE && act != SVDX_ACT_GELU))
    return svdx_fail(SVDX_E_BADARG, "splitk_epilogue: bad arguments");
  splitk_epilogue_kernel<<<nblocks(rows * (cols / 8)), 256, 0, ST(stream)>>>(ws, ldw, reinterpret_cast<bf16*>(out), ldo, rows, cols, bias, rowbias,
                                                                            rowbias_div, ldrb, reinterpret_cast<const bf16*>(res1), ldr1,
                                                                            reinterpret_cast<const bf16*>(res2), ldr2, scales, act);
  SVDX_CHECK_LAUNCH("splitk_epilogue");
  return SVDX_OK;
}

extern "C" int svdx_splitk_epilogue(float* ws, int64_t ldw, void* out, int64_t ldo, int64_t rows, int32_t cols, const float* bias,
                                    const float* rowbias, int32_t rowbias_div, int64_t ldrb, const void* res1, int64_t ldr1,
                                    const void* res2, int64_t ldr2, const float* scales, void* stream) {
  return svdx_splitk_epilogue_act(ws, ldw, out, ldo, rows, cols, bias, rowbias, rowbias_div, ldrb, res1, ldr1, res2, ldr2, scales,
                                  SVDX_ACT_NONE, stream);
}

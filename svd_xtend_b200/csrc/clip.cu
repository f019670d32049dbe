// CLIP image preprocessing + ViT patchify in one launch (svdx_clip_pixels, include/svd_xtend_b200.h).
//
// encode_image (train_svd.py:857-876) runs _resize_with_antialiasing (a separable Gaussian blur with reflect padding, then
// bicubic align_corners=True resampling to 224 x 224), (x + 1) / 2, and the CLIPImageProcessor normalisation, and the ViT then
// cuts the 224 x 224 image into 16 x 16 patches of 14 x 14 pixels for its patch-embedding convolution (a GEMM over K = 588).
// All of it is linear up to the final affine step, so one CTA produces one output image row (b, c, oy) directly:
//   1. vertical pass: the 4 bicubic source rows of oy, each blurred along H (ky taps, reflect padding), weighted and summed
//      into one row of W values in shared memory (coalesced reads of 4 * ky input rows);
//   2. horizontal pass: for each of the 224 output columns, the 4 bicubic source columns, each blurred along W, from that row;
//   3. (v + 1) / 2, (v - mean_c) / std_c, rounded to bf16 and stored at its (patch row, (c, ky, kx)) position of the patch matrix.
// The blur and resampling are reordered (vertical first) relative to the reference; both are linear, so the result is the same
// up to rounding. resize = 0 is the patchify of an already normalised 224 x 224 input.
// The resize is computed in float64 (a few M FMAs per image, far from any limit of the chip): in float32 the bicubic source
// coordinate dst * (in - 1) / 223 is off by up to ~3e-5 pixels at the far edge (~1e-4 in the value), and the subtraction of
// the channel mean leaves outputs near zero with few correct bits, so a float32 kernel is not within one bf16 ulp of the
// exact resize. In float64 the stored bf16 is the correctly rounded exact value except at rounding ties.
#include "common.cuh"
#include "../../include/svd_xtend_b200.h"
#include "host_util.h"

namespace svdx {

constexpr int CLIP_OUT = 224;
constexpr int CLIP_PATCH = 14;
constexpr int CLIP_K = 3 * CLIP_PATCH * CLIP_PATCH;   // 588
constexpr int CLIP_KP = 592;
constexpr int CLIP_MAX_W = 6144;                      // float64 row in the default 48 KB of dynamic shared memory

struct ClipP {
  const void* x;
  int dtype, H, W, resize, ky, kx;
  double wy[SVDX_CLIP_MAX_TAPS], wx[SVDX_CLIP_MAX_TAPS];
  double mean[3], std[3];
  double sy, sx;   // bicubic source scale (in - 1) / (224 - 1)
  bf16* out;
  long long ldo;
};

SVDX_DEVINL double clip_load(const void* x, int dtype, long long i) {
  if (dtype == 0) return (double)__ldg(reinterpret_cast<const float*>(x) + i);
  if (dtype == 1) return (double)__bfloat162float(reinterpret_cast<const bf16*>(x)[i]);
  return (double)__half2float(reinterpret_cast<const __half*>(x)[i]);
}
SVDX_DEVINL int reflect_idx(int i, int n) { return i < 0 ? -i : (i >= n ? 2 * (n - 1) - i : i); }
SVDX_DEVINL int clamp_idx(int i, int n) { return i < 0 ? 0 : (i >= n ? n - 1 : i); }

// PyTorch's bicubic weights (A = -0.75) of the 4 neighbours floor(src) - 1 .. floor(src) + 2
SVDX_DEVINL void cubic_coeffs(double t, double (&c)[4]) {
  const double A = -0.75;
  auto cc1 = [&](double x) { return ((A + 2.0) * x - (A + 3.0)) * x * x + 1.0; };
  auto cc2 = [&](double x) { return ((A * x - 5.0 * A) * x + 8.0 * A) * x - 4.0 * A; };
  c[0] = cc2(t + 1.0);
  c[1] = cc1(t);
  c[2] = cc1(1.0 - t);
  c[3] = cc2(2.0 - t);
}

__global__ void __launch_bounds__(256) clip_pixels_kernel(const ClipP p) {
  extern __shared__ double row[];
  const int oy = blockIdx.x, c = blockIdx.y, b = blockIdx.z;
  const long long plane = ((long long)b * 3 + c) * p.H * p.W;
  const long long orow0 = (long long)b * 256 + (oy / CLIP_PATCH) * 16;
  const int kcol0 = c * CLIP_PATCH * CLIP_PATCH + (oy % CLIP_PATCH) * CLIP_PATCH;
  if (c == 0 && oy % CLIP_PATCH == 0 && threadIdx.x < 16 * (CLIP_KP - CLIP_K))   // zero columns 588 .. 591 of this patch row
    p.out[(orow0 + threadIdx.x / 4) * p.ldo + CLIP_K + (threadIdx.x & 3)] = __float2bfloat16(0.f);
  if (!p.resize) {
    for (int ox = threadIdx.x; ox < CLIP_OUT; ox += blockDim.x) {
      const double v = clip_load(p.x, p.dtype, plane + (long long)oy * p.W + ox);
      p.out[(orow0 + ox / CLIP_PATCH) * p.ldo + kcol0 + ox % CLIP_PATCH] = __double2bfloat16(v);
    }
    return;
  }
  // 1. vertical: bicubic rows of oy, each blurred along H
  const double ry = p.sy * (double)oy;
  const int iy = (int)floor(ry);
  double cy[4];
  cubic_coeffs(ry - (double)iy, cy);
  const int py = (p.ky - 1) / 2, px = (p.kx - 1) / 2;
  for (int xx = threadIdx.x; xx < p.W; xx += blockDim.x) {
    double acc = 0.0;
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      const int ya = clamp_idx(iy - 1 + a, p.H);
      double s = 0.0;
      for (int i = 0; i < p.ky; ++i) s = fma(p.wy[i], clip_load(p.x, p.dtype, plane + (long long)reflect_idx(ya + i - py, p.H) * p.W + xx), s);
      acc = fma(cy[a], s, acc);
    }
    row[xx] = acc;
  }
  __syncthreads();
  // 2. horizontal, 3. normalise and place
  const double mean = p.mean[c], std = p.std[c];
  for (int ox = threadIdx.x; ox < CLIP_OUT; ox += blockDim.x) {
    const double rx = p.sx * (double)ox;
    const int ix = (int)floor(rx);
    double cx[4];
    cubic_coeffs(rx - (double)ix, cx);
    double acc = 0.0;
#pragma unroll
    for (int a = 0; a < 4; ++a) {
      const int xa = clamp_idx(ix - 1 + a, p.W);
      double s = 0.0;
      for (int j = 0; j < p.kx; ++j) s = fma(p.wx[j], row[reflect_idx(xa + j - px, p.W)], s);
      acc = fma(cx[a], s, acc);
    }
    const double v = ((acc + 1.0) * 0.5 - mean) / std;
    p.out[(orow0 + ox / CLIP_PATCH) * p.ldo + kcol0 + ox % CLIP_PATCH] = __double2bfloat16(v);
  }
}

}  // namespace svdx

using namespace svdx;

extern "C" int svdx_clip_pixels(const SvdxClipPixels* d, void* stream) {
  if (!d || !d->x || !d->out) return svdx_fail(SVDX_E_BADARG, "clip_pixels: null pointer");
  if (d->dtype < 0 || d->dtype > 2 || d->B <= 0 || d->B > 65535 || d->ldo < CLIP_KP || d->ldo % 8)
    return svdx_fail(SVDX_E_BADARG, "clip_pixels: bad arguments (dtype code 0/1/2, 1 <= B <= 65535, ldo >= 592, ldo %% 8 == 0)");
  ClipP p;
  memset(&p, 0, sizeof(p));
  if (d->resize) {
    if (d->H < CLIP_PATCH || d->W < CLIP_PATCH || d->W > CLIP_MAX_W)
      return svdx_fail(SVDX_E_BADARG, "clip_pixels: resize needs 14 <= H and 14 <= W <= 6144");
    if (d->ky < 1 || d->kx < 1 || d->ky > SVDX_CLIP_MAX_TAPS || d->kx > SVDX_CLIP_MAX_TAPS || !(d->ky & 1) || !(d->kx & 1) ||
        (d->ky - 1) / 2 >= d->H || (d->kx - 1) / 2 >= d->W)
      return svdx_fail(SVDX_E_BADARG, "clip_pixels: blur taps must be odd counts <= 31 with padding smaller than the image");
    if (!(d->std[0] > 0.0) || !(d->std[1] > 0.0) || !(d->std[2] > 0.0)) return svdx_fail(SVDX_E_BADARG, "clip_pixels: std must be > 0");
    p.ky = d->ky; p.kx = d->kx;
    for (int i = 0; i < d->ky; ++i) p.wy[i] = d->wy[i];
    for (int i = 0; i < d->kx; ++i) p.wx[i] = d->wx[i];
    for (int i = 0; i < 3; ++i) { p.mean[i] = d->mean[i]; p.std[i] = d->std[i]; }
    p.sy = (double)(d->H - 1) / (double)(CLIP_OUT - 1);
    p.sx = (double)(d->W - 1) / (double)(CLIP_OUT - 1);
  } else if (d->H != CLIP_OUT || d->W != CLIP_OUT) {
    return svdx_fail(SVDX_E_BADARG, "clip_pixels: resize = 0 needs 224 x 224 input");
  }
  p.x = d->x; p.dtype = d->dtype; p.H = d->H; p.W = d->W; p.resize = d->resize ? 1 : 0;
  p.out = reinterpret_cast<bf16*>(d->out); p.ldo = d->ldo;
  const size_t smem = p.resize ? (size_t)p.W * sizeof(double) : 0;
  clip_pixels_kernel<<<dim3(CLIP_OUT, 3, (unsigned)d->B), 256, smem, reinterpret_cast<cudaStream_t>(stream)>>>(p);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return svdx_fail_cuda(e, "clip_pixels: launch");
  return SVDX_OK;
}

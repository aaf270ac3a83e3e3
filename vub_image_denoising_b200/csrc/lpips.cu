// lpips.cu — the non-GEMM kernels of LPIPS (lpips 0.1, net='alex'; evaluate_Unet_diffusion/evaluate_model.py:46-71).
//   patch gathers  : im2col of AlexNet's conv1 (11x11/s4/p2, from the fp32 NCHW image pair with the ScalingLayer
//                    affine fused in) and conv2 (5x5/p2, from the pooled NHWC 16-bit map); the convolutions then run
//                    as b200dn_igemm MODE_CONV1X1 GEMMs over these rows
//   max-pool 3x3/s2: floor mode, no padding, on NHWC 16-bit planes
//   head           : per tap, pixel: unit-normalise the two feature vectors over channels, weight the squared
//                    difference with lin{l}, then the spatial mean per tap and the sum over taps
// Storage is bf16 (one plane, or hi + lo planes for the two-plane precisions); patch rows are (ky, kx, ci)-ordered and
// zero padded to kpad columns.  The head is two-pass and atomics-free like metrics.cu: one fp64 partial per block, then
// a fixed-order sum per image, so the result is bit-reproducible and an image's value does not depend on the batch.
#include <string.h>

#include "perceptual.cuh"

namespace b200dn {

namespace {

using namespace perceptual;

__device__ __forceinline__ float bf16x2_val(uint32_t hi, uint32_t lo, bool lo_half, bool two) {
  const float h = lo_half ? bf16_lo(hi) : bf16_hi(hi);
  return two ? h + (lo_half ? bf16_lo(lo) : bf16_hi(lo)) : h;
}

// ---------------------------------------------------------------- conv1 patches from the fp32 NCHW image pair
// Work item = 8 consecutive K columns of one output pixel of image b (b < N: in0[b], else in1[b - N]).
// x' = (x - shift[c]) / scale[c] (x = 2x - 1 first with normalize), the ScalingLayer's fp32 operation order; taps
// outside the image are 0: the conv pads the SCALED image.
__global__ void __launch_bounds__(LP_THREADS) gather_image_kernel(
    const float* __restrict__ in0, const float* __restrict__ in1, int N, int C, int H, int W,
    const float* __restrict__ shift, const float* __restrict__ scale, int normalize, int kh, int kw, int stride,
    int pad, int Ho, int Wo, int kpad, int two, uint16_t* __restrict__ out0, uint16_t* __restrict__ out1) {
  const int K = kh * kw * C;
  const int k8n = kpad / 8;
  const int64_t n_items = static_cast<int64_t>(2 * N) * Ho * Wo * k8n;
  const int64_t step = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n_items; i += step) {
    const int k0 = static_cast<int>(i % k8n) * 8;
    const int64_t pix = i / k8n;
    const int ox = static_cast<int>(pix % Wo);
    const int oy = static_cast<int>((pix / Wo) % Ho);
    const int b = static_cast<int>(pix / (static_cast<int64_t>(Wo) * Ho));
    const float* src = b < N ? in0 + static_cast<int64_t>(b) * C * H * W : in1 + static_cast<int64_t>(b - N) * C * H * W;
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int k = k0 + j;
      float x = 0.f;
      if (k < K) {
        const int ky = k / (kw * C), rem = k - ky * (kw * C);
        const int kx = rem / C, c = rem - kx * C;
        const int iy = oy * stride - pad + ky, ix = ox * stride - pad + kx;
        if (iy >= 0 && iy < H && ix >= 0 && ix < W) {
          x = __ldg(src + (static_cast<int64_t>(c) * H + iy) * W + ix);
          if (normalize) x = __fsub_rn(__fmul_rn(2.f, x), 1.f);
          x = __fdiv_rn(__fsub_rn(x, __ldg(shift + c)), __ldg(scale + c));
        }
      }
      v[j] = x;
    }
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      hi[q] = pack_bf16x2(v[2 * q], v[2 * q + 1]);
      lo[q] = pack_bf16x2(v[2 * q] - bf16_lo(hi[q]), v[2 * q + 1] - bf16_hi(hi[q]));
    }
    const int64_t o = pix * kpad + k0;
    *reinterpret_cast<uint4*>(out0 + o) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    if (two) *reinterpret_cast<uint4*>(out1 + o) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
  }
}

// ---------------------------------------------------------------- patches from NHWC 16-bit planes
// Work item = one 8-channel chunk (16 bytes per plane) of one (ky, kx) tap of one output pixel.
__global__ void __launch_bounds__(LP_THREADS) gather_nhwc_kernel(
    const uint16_t* __restrict__ in0, const uint16_t* __restrict__ in1, int B, int H, int W, int C, int kh, int kw,
    int stride, int pad, int Ho, int Wo, int kpad, int two, uint16_t* __restrict__ out0, uint16_t* __restrict__ out1) {
  const int k8n = kpad / 8, c8n = C / 8, k8_used = kh * kw * c8n;
  const int64_t n_items = static_cast<int64_t>(B) * Ho * Wo * k8n;
  const int64_t step = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n_items; i += step) {
    const int k8 = static_cast<int>(i % k8n);
    const int64_t pix = i / k8n;
    uint4 h = make_uint4(0, 0, 0, 0), l = h;
    if (k8 < k8_used) {
      const int ox = static_cast<int>(pix % Wo);
      const int oy = static_cast<int>((pix / Wo) % Ho);
      const int b = static_cast<int>(pix / (static_cast<int64_t>(Wo) * Ho));
      const int ky = k8 / (kw * c8n), rem = k8 - ky * (kw * c8n);
      const int kx = rem / c8n, c8 = rem - kx * c8n;
      const int iy = oy * stride - pad + ky, ix = ox * stride - pad + kx;
      if (iy >= 0 && iy < H && ix >= 0 && ix < W) {
        const int64_t s = ((static_cast<int64_t>(b) * H + iy) * W + ix) * C + c8 * 8;
        h = __ldg(reinterpret_cast<const uint4*>(in0 + s));
        if (two) l = __ldg(reinterpret_cast<const uint4*>(in1 + s));
      }
    }
    const int64_t o = pix * kpad + k8 * 8;
    *reinterpret_cast<uint4*>(out0 + o) = h;
    if (two) *reinterpret_cast<uint4*>(out1 + o) = l;
  }
}

// ---------------------------------------------------------------- max-pool 3x3 / stride 2
// Work item = one 8-channel chunk of one output pixel.  With two planes the max is taken over the value hi + lo (exact
// in fp32) and the winning (hi, lo) pair is copied: the per-plane maxima could come from different taps.  Ties keep the
// first tap in (ky, kx) order, as the values are equal.
__global__ void __launch_bounds__(LP_THREADS) maxpool_kernel(const uint16_t* __restrict__ in0,
                                                             const uint16_t* __restrict__ in1, int B, int H, int W,
                                                             int C, int Ho, int Wo, int two, uint16_t* __restrict__ out0,
                                                             uint16_t* __restrict__ out1) {
  const int c8n = C / 8;
  const int64_t n_items = static_cast<int64_t>(B) * Ho * Wo * c8n;
  const int64_t step = static_cast<int64_t>(gridDim.x) * blockDim.x;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x; i < n_items; i += step) {
    const int c8 = static_cast<int>(i % c8n);
    const int64_t pix = i / c8n;
    const int ox = static_cast<int>(pix % Wo);
    const int oy = static_cast<int>((pix / Wo) % Ho);
    const int b = static_cast<int>(pix / (static_cast<int64_t>(Wo) * Ho));
    float best[8];
    alignas(16) uint16_t bh[8], bl[8];
#pragma unroll
    for (int t = 0; t < 9; ++t) {
      const int ky = t / 3, kx = t - ky * 3;
      const int64_t s = ((static_cast<int64_t>(b) * H + 2 * oy + ky) * W + 2 * ox + kx) * C + c8 * 8;
      alignas(16) uint16_t h[8], l[8];
      *reinterpret_cast<uint4*>(h) = __ldg(reinterpret_cast<const uint4*>(in0 + s));
      *reinterpret_cast<uint4*>(l) = two ? __ldg(reinterpret_cast<const uint4*>(in1 + s)) : make_uint4(0, 0, 0, 0);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float v = bf16_lo(h[j]) + bf16_lo(l[j]);
        if (t == 0 || v > best[j]) best[j] = v, bh[j] = h[j], bl[j] = l[j];
      }
    }
    const int64_t o = pix * C + c8 * 8;
    *reinterpret_cast<uint4*>(out0 + o) = *reinterpret_cast<const uint4*>(bh);
    if (two) *reinterpret_cast<uint4*>(out1 + o) = *reinterpret_cast<const uint4*>(bl);
  }
}

// ---------------------------------------------------------------- LPIPS head
constexpr int HEAD_MAX_TAPS = 8;
constexpr int HEAD_MAX_C = 512;              // 8-channel chunks per lane: HEAD_MAX_C / 256
constexpr int HEAD_PIX_PER_BLOCK = 64;       // 8 warps x 8 pixels: the block partition depends on H x W only
constexpr float HEAD_EPS = 1e-10f;           // lpips.normalize_tensor: x / (sqrt(sum x^2) + eps)

struct HeadParams {
  const uint16_t* f0[HEAD_MAX_TAPS];
  const uint16_t* f1[HEAD_MAX_TAPS];
  const float* w[HEAD_MAX_TAPS];
  int hw[HEAD_MAX_TAPS], C[HEAD_MAX_TAPS];
  int blk0[HEAD_MAX_TAPS + 1];               // first block of each tap in an image's block range
  int n_taps, N, two;
};

// 8 channels of one pixel of one image as fp32 (hi + lo)
__device__ __forceinline__ void load8(const uint16_t* p0, const uint16_t* p1, int64_t off, bool two, float (&v)[8]) {
  const uint4 h4 = __ldg(reinterpret_cast<const uint4*>(p0 + off));
  const uint4 l4 = two ? __ldg(reinterpret_cast<const uint4*>(p1 + off)) : make_uint4(0, 0, 0, 0);
  const uint32_t h[4] = {h4.x, h4.y, h4.z, h4.w}, l[4] = {l4.x, l4.y, l4.z, l4.w};
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    v[2 * q] = bf16x2_val(h[q], l[q], true, two);
    v[2 * q + 1] = bf16x2_val(h[q], l[q], false, two);
  }
}

// grid = (blocks of all taps, N).  Warp = one pixel at a time, lane = 8-channel chunks lane, lane + 32.  Image n's
// features are batch entry n, its partner's entry N + n; both go through identical code, so d(a, b) == d(b, a) bit for
// bit and d(a, a) == 0.
__global__ void __launch_bounds__(LP_THREADS) lpips_head_kernel(const __grid_constant__ HeadParams p,
                                                                double* __restrict__ partial) {
  __shared__ double red[LP_THREADS / 32];
  const int n = blockIdx.y, blk = blockIdx.x;
  int l = 0;
  while (l + 1 < p.n_taps && blk >= p.blk0[l + 1]) ++l;
  const int C = p.C[l], c8n = C / 8, hw = p.hw[l];
  const bool two = p.two != 0;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t img0 = static_cast<int64_t>(n) * hw * C, img1 = static_cast<int64_t>(p.N + n) * hw * C;
  double acc = 0.0;
  for (int i = 0; i < HEAD_PIX_PER_BLOCK / (LP_THREADS / 32); ++i) {
    const int pix = (blk - p.blk0[l]) * HEAD_PIX_PER_BLOCK + i * (LP_THREADS / 32) + warp;
    if (pix >= hw) break;
    float a[HEAD_MAX_C / 256][8], b[HEAD_MAX_C / 256][8];
    float s0 = 0.f, s1 = 0.f;
#pragma unroll
    for (int r = 0; r < HEAD_MAX_C / 256; ++r) {
      const int c8 = lane + 32 * r;
      if (c8 < c8n) {
        load8(p.f0[l], p.f1[l], img0 + static_cast<int64_t>(pix) * C + c8 * 8, two, a[r]);
        load8(p.f0[l], p.f1[l], img1 + static_cast<int64_t>(pix) * C + c8 * 8, two, b[r]);
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) a[r][j] = b[r][j] = 0.f;
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        s0 = fmaf(a[r][j], a[r][j], s0);
        s1 = fmaf(b[r][j], b[r][j], s1);
      }
    }
    s0 = warp_sum_f(s0);
    s1 = warp_sum_f(s1);
    const float den0 = __fadd_rn(__fsqrt_rn(s0), HEAD_EPS), den1 = __fadd_rn(__fsqrt_rn(s1), HEAD_EPS);
    float d = 0.f;
#pragma unroll
    for (int r = 0; r < HEAD_MAX_C / 256; ++r) {
      const int c8 = lane + 32 * r;
      if (c8 < c8n) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float e = __fsub_rn(__fdiv_rn(a[r][j], den0), __fdiv_rn(b[r][j], den1));
          d = fmaf(__ldg(p.w[l] + c8 * 8 + j), __fmul_rn(e, e), d);
        }
      }
    }
    acc += static_cast<double>(warp_sum_f(d));   // identical in every lane
  }
  if (lane == 0) red[warp] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
#pragma unroll
    for (int k = 0; k < LP_THREADS / 32; ++k) t += red[k];
    partial[static_cast<int64_t>(n) * p.blk0[p.n_taps] + blk] = t;
  }
}

// One warp per image: per tap (in order) the fixed-order sum of its block partials over H x W, then the sum over taps.
__global__ void __launch_bounds__(128) lpips_finish_kernel(const __grid_constant__ HeadParams p,
                                                           const double* __restrict__ partial, float* __restrict__ out) {
  const int n = blockIdx.x * 4 + (threadIdx.x >> 5);
  if (n >= p.N) return;
  const int lane = threadIdx.x & 31;
  const double* q = partial + static_cast<int64_t>(n) * p.blk0[p.n_taps];
  double total = 0.0;
  for (int l = 0; l < p.n_taps; ++l) {
    double s = 0.0;
    for (int k = p.blk0[l] + lane; k < p.blk0[l + 1]; k += 32) s += q[k];
    total += warp_sum_d(s) / static_cast<double>(p.hw[l]);
  }
  if (lane == 0) out[n] = static_cast<float>(total);
}

int head_params(const b200dn_lpips_tap* taps, int n_taps, int N, int prec, HeadParams& p) {
  B200DN_CHECK_ARG(taps && n_taps >= 1 && n_taps <= HEAD_MAX_TAPS, "lpips_head: 1..%d taps", HEAD_MAX_TAPS);
  B200DN_CHECK_ARG(N >= 1 && N <= 65535, "lpips_head: 1..65535 image pairs");
  B200DN_CHECK_ARG(bf16_prec(prec), "lpips_head: prec %d: only the bf16-stored precisions are supported", prec);
  memset(&p, 0, sizeof(p));
  p.n_taps = n_taps, p.N = N, p.two = two_planes(prec) ? 1 : 0;
  int64_t blocks = 0;
  for (int l = 0; l < n_taps; ++l) {
    const b200dn_lpips_tap& t = taps[l];
    B200DN_CHECK_ARG(t.feat[0] && (!p.two || t.feat[1]) && t.weight, "lpips_head: tap %d: null pointer", l);
    B200DN_CHECK_ARG(((reinterpret_cast<uintptr_t>(t.feat[0]) | reinterpret_cast<uintptr_t>(t.feat[1])) & 15) == 0,
                     "lpips_head: tap %d: feature planes must be 16-byte aligned", l);
    B200DN_CHECK_ARG(t.H > 0 && t.W > 0 && t.C > 0 && t.C % 8 == 0 && t.C <= HEAD_MAX_C,
                     "lpips_head: tap %d: H, W > 0 and C a multiple of 8 up to %d (got %d x %d x %d)", l, HEAD_MAX_C,
                     t.H, t.W, t.C);
    p.f0[l] = static_cast<const uint16_t*>(t.feat[0]);
    p.f1[l] = static_cast<const uint16_t*>(t.feat[1]);
    p.w[l] = t.weight;
    p.hw[l] = t.H * t.W;
    p.C[l] = t.C;
    p.blk0[l] = static_cast<int>(blocks);
    blocks += cdiv64(static_cast<int64_t>(t.H) * t.W, HEAD_PIX_PER_BLOCK);
    B200DN_CHECK_ARG(blocks < (1 << 30), "lpips_head: too many pixels");
  }
  p.blk0[n_taps] = static_cast<int>(blocks);
  return 0;
}

}  // namespace
}  // namespace b200dn

extern "C" int b200dn_patch_gather_image(const float* in0, const float* in1, int N, int C, int H, int W,
                                         const float* shift, const float* scale, int normalize, int kh, int kw,
                                         int stride, int pad, int kpad, int prec, void* out0, void* out1,
                                         void* stream) {
  using namespace b200dn;
  B200DN_CHECK_ARG(in0 && in1 && shift && scale && out0, "patch_gather_image: null pointer");
  B200DN_CHECK_ARG(bf16_prec(prec), "patch_gather_image: prec %d: only the bf16-stored precisions are supported", prec);
  B200DN_CHECK_ARG(!two_planes(prec) || out1, "patch_gather_image: prec %d needs the lo output plane", prec);
  B200DN_CHECK_ARG(N > 0 && C > 0 && H > 0 && W > 0 && kh > 0 && kw > 0 && stride > 0 && pad >= 0,
                   "patch_gather_image: bad shape");
  B200DN_CHECK_ARG(H + 2 * pad >= kh && W + 2 * pad >= kw, "patch_gather_image: kernel larger than the padded image");
  B200DN_CHECK_ARG(kpad % 8 == 0 && kpad >= kh * kw * C, "patch_gather_image: kpad %d must be a multiple of 8 >= %d",
                   kpad, kh * kw * C);
  B200DN_CHECK_ARG(((reinterpret_cast<uintptr_t>(out0) | reinterpret_cast<uintptr_t>(out1)) & 15) == 0,
                   "patch_gather_image: output planes must be 16-byte aligned");
  if (int rc = require_sm100()) return rc;
  const int Ho = (H + 2 * pad - kh) / stride + 1, Wo = (W + 2 * pad - kw) / stride + 1;
  const int grid = lp_grid(static_cast<int64_t>(2 * N) * Ho * Wo * (kpad / 8));
  if (grid <= 0) return B200DN_E_CUDA;
  gather_image_kernel<<<grid, LP_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(
      in0, in1, N, C, H, W, shift, scale, normalize, kh, kw, stride, pad, Ho, Wo, kpad, two_planes(prec) ? 1 : 0,
      static_cast<uint16_t*>(out0), static_cast<uint16_t*>(out1));
  B200DN_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int b200dn_patch_gather(const void* in_hi, const void* in_lo, int B, int H, int W, int C, int kh, int kw,
                                   int stride, int pad, int kpad, int prec, void* out0, void* out1, void* stream) {
  using namespace b200dn;
  B200DN_CHECK_ARG(in_hi && out0, "patch_gather: null pointer");
  B200DN_CHECK_ARG(bf16_prec(prec), "patch_gather: prec %d: only the bf16-stored precisions are supported", prec);
  B200DN_CHECK_ARG(!two_planes(prec) || (in_lo && out1), "patch_gather: prec %d needs the lo planes", prec);
  B200DN_CHECK_ARG(B > 0 && H > 0 && W > 0 && C > 0 && C % 8 == 0 && kh > 0 && kw > 0 && stride > 0 && pad >= 0,
                   "patch_gather: bad shape (C must be a multiple of 8)");
  B200DN_CHECK_ARG(H + 2 * pad >= kh && W + 2 * pad >= kw, "patch_gather: kernel larger than the padded image");
  B200DN_CHECK_ARG(kpad % 8 == 0 && kpad >= kh * kw * C, "patch_gather: kpad %d must be a multiple of 8 >= %d", kpad,
                   kh * kw * C);
  B200DN_CHECK_ARG(((reinterpret_cast<uintptr_t>(in_hi) | reinterpret_cast<uintptr_t>(in_lo) |
                     reinterpret_cast<uintptr_t>(out0) | reinterpret_cast<uintptr_t>(out1)) & 15) == 0,
                   "patch_gather: planes must be 16-byte aligned");
  if (int rc = require_sm100()) return rc;
  const int Ho = (H + 2 * pad - kh) / stride + 1, Wo = (W + 2 * pad - kw) / stride + 1;
  const int grid = lp_grid(static_cast<int64_t>(B) * Ho * Wo * (kpad / 8));
  if (grid <= 0) return B200DN_E_CUDA;
  gather_nhwc_kernel<<<grid, LP_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const uint16_t*>(in_hi), static_cast<const uint16_t*>(in_lo), B, H, W, C, kh, kw, stride, pad, Ho,
      Wo, kpad, two_planes(prec) ? 1 : 0, static_cast<uint16_t*>(out0), static_cast<uint16_t*>(out1));
  B200DN_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int b200dn_maxpool3x3s2(const void* in_hi, const void* in_lo, int B, int H, int W, int C, int prec,
                                   void* out0, void* out1, void* stream) {
  using namespace b200dn;
  B200DN_CHECK_ARG(in_hi && out0, "maxpool3x3s2: null pointer");
  B200DN_CHECK_ARG(bf16_prec(prec), "maxpool3x3s2: prec %d: only the bf16-stored precisions are supported", prec);
  B200DN_CHECK_ARG(!two_planes(prec) || (in_lo && out1), "maxpool3x3s2: prec %d needs the lo planes", prec);
  B200DN_CHECK_ARG(B > 0 && H >= 3 && W >= 3 && C > 0 && C % 8 == 0,
                   "maxpool3x3s2: needs H, W >= 3 and C a multiple of 8 (got %d x %d x %d)", H, W, C);
  B200DN_CHECK_ARG(((reinterpret_cast<uintptr_t>(in_hi) | reinterpret_cast<uintptr_t>(in_lo) |
                     reinterpret_cast<uintptr_t>(out0) | reinterpret_cast<uintptr_t>(out1)) & 15) == 0,
                   "maxpool3x3s2: planes must be 16-byte aligned");
  if (int rc = require_sm100()) return rc;
  const int Ho = (H - 3) / 2 + 1, Wo = (W - 3) / 2 + 1;
  const int grid = lp_grid(static_cast<int64_t>(B) * Ho * Wo * (C / 8));
  if (grid <= 0) return B200DN_E_CUDA;
  maxpool_kernel<<<grid, LP_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const uint16_t*>(in_hi), static_cast<const uint16_t*>(in_lo), B, H, W, C, Ho, Wo,
      two_planes(prec) ? 1 : 0, static_cast<uint16_t*>(out0), static_cast<uint16_t*>(out1));
  B200DN_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int64_t b200dn_lpips_head_workspace_bytes(const b200dn_lpips_tap* taps, int n_taps, int N) {
  b200dn::HeadParams p;
  if (b200dn::head_params(taps, n_taps, N, B200DN_PREC_BF16, p)) return 0;
  return static_cast<int64_t>(N) * p.blk0[n_taps] * static_cast<int64_t>(sizeof(double));
}

extern "C" int b200dn_lpips_head(const b200dn_lpips_tap* taps, int n_taps, int N, int prec, float* out,
                                 void* workspace, int64_t workspace_bytes, void* stream) {
  using namespace b200dn;
  HeadParams p;
  if (int rc = head_params(taps, n_taps, N, prec, p)) return rc;
  B200DN_CHECK_ARG(out, "lpips_head: null output");
  B200DN_CHECK_ARG(workspace && (reinterpret_cast<uintptr_t>(workspace) & 7) == 0 &&
                       workspace_bytes >= static_cast<int64_t>(N) * p.blk0[n_taps] * static_cast<int64_t>(sizeof(double)),
                   "lpips_head: workspace of b200dn_lpips_head_workspace_bytes() bytes (8-byte aligned) required");
  if (int rc = require_sm100()) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  double* partial = static_cast<double*>(workspace);
  lpips_head_kernel<<<dim3(static_cast<unsigned>(p.blk0[n_taps]), static_cast<unsigned>(N)), LP_THREADS, 0, s>>>(p, partial);
  B200DN_CUDA(cudaGetLastError());
  lpips_finish_kernel<<<static_cast<unsigned>(cdiv(N, 4)), 128, 0, s>>>(p, partial, out);
  B200DN_CUDA(cudaGetLastError());
  return 0;
}

// dists.cu — the non-GEMM kernels of DISTS (DISTS_pytorch 0.1, DISTS_pt.py; evaluate_Unet_diffusion/evaluate_model.py:46-71).
//   L2 pooling 3x3/s2: sqrt(conv2d(x^2, filter, stride 2, padding 1, groups C) + 1e-12) on NHWC 16-bit planes, the
//                      depthwise taps read from the module's filter buffer
//   head             : per image pair, stage and channel the moments sum x, y, x^2, y^2, xy over H x W, then
//                      S1 = (2 mx my + c1) / (mx^2 + my^2 + c1), S2 = (2 cov + c2) / (vx + vy + c2) (population
//                      moments), score = 1 - sum_c (alpha_c S1 + beta_c S2) / (sum alpha + sum beta)
// The VGG16 convolutions run on b200dn_igemm (conv1_1 as a MODE_CONV1X1 GEMM over the rows of
// b200dn_patch_gather_image, the rest MODE_CONV3X3).  The head is two-pass and atomics-free like lpips.cu: fp64 moment
// partials, one per (channel, pixel chunk), then a fixed-order sum per image pair, so the score is bit-reproducible, a
// pair's score does not depend on the batch, and D(x, y) == D(y, x) bit for bit (x and y go through identical code and
// every operation combining them is commutative).
#include <string.h>

#include "perceptual.cuh"

namespace b200dn {

namespace {

using namespace perceptual;

// ---------------------------------------------------------------- L2 pooling 3x3 / stride 2 / padding 1
// Work item = one 8-channel chunk of one output pixel.  fp32: v = hi + lo, sum over the taps in (ky, kx) order of
// filter * v^2, taps outside the image are 0; stored as hi = bf16(o), lo = bf16(o - hi).
__global__ void __launch_bounds__(LP_THREADS) l2pool_kernel(const uint16_t* __restrict__ in0,
                                                            const uint16_t* __restrict__ in1, int B, int H, int W,
                                                            int C, const float* __restrict__ filter, int Ho, int Wo,
                                                            int two, uint16_t* __restrict__ out0,
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
    const float* f = filter + c8 * 8 * 9;
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = 0.f;
#pragma unroll
    for (int t = 0; t < 9; ++t) {
      const int ky = t / 3, kx = t - ky * 3;
      const int iy = 2 * oy - 1 + ky, ix = 2 * ox - 1 + kx;
      if (iy < 0 || iy >= H || ix < 0 || ix >= W) continue;
      const int64_t s = ((static_cast<int64_t>(b) * H + iy) * W + ix) * C + c8 * 8;
      alignas(16) uint16_t h[8], l[8];
      *reinterpret_cast<uint4*>(h) = __ldg(reinterpret_cast<const uint4*>(in0 + s));
      *reinterpret_cast<uint4*>(l) = two ? __ldg(reinterpret_cast<const uint4*>(in1 + s)) : make_uint4(0, 0, 0, 0);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float v = __fadd_rn(bf16_lo(h[j]), bf16_lo(l[j]));
        acc[j] = __fmaf_rn(__ldg(f + j * 9 + t), __fmul_rn(v, v), acc[j]);
      }
    }
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float a = __fsqrt_rn(__fadd_rn(acc[2 * q], 1e-12f)), b2 = __fsqrt_rn(__fadd_rn(acc[2 * q + 1], 1e-12f));
      hi[q] = pack_bf16x2(a, b2);
      lo[q] = pack_bf16x2(a - bf16_lo(hi[q]), b2 - bf16_hi(hi[q]));
    }
    const int64_t o = pix * C + c8 * 8;
    *reinterpret_cast<uint4*>(out0 + o) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    if (two) *reinterpret_cast<uint4*>(out1 + o) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
  }
}

// ---------------------------------------------------------------- DISTS head
constexpr int DS_MAX_STAGES = 8;             // stage 0 (the image) + up to 7 feature stages
constexpr int DS_PIX = 1024;                 // pixels per chunk: the chunk partition depends on H x W only
constexpr int DS_GROUP = 64;                 // channels per block of a feature stage (2 per lane)
constexpr double DS_C1 = 1e-6, DS_C2 = 1e-6;

struct DistsParams {
  const float* img0;                         // stage 0: fp32 NCHW [N, 3, H, W], in0 and in1
  const float* img1;
  const uint16_t* f0[DS_MAX_STAGES];         // stages >= 1: NHWC [2N, H_k, W_k, C_k] hi, lo planes
  const uint16_t* f1[DS_MAX_STAGES];
  const float* alpha;                        // [c0[n_stages]] each, in stage order
  const float* beta;
  int hw[DS_MAX_STAGES], C[DS_MAX_STAGES], chunks[DS_MAX_STAGES];
  int blk0[DS_MAX_STAGES + 1];               // first block of each stage in a pair's block range
  int slot0[DS_MAX_STAGES + 1];              // first (channel, chunk) slot of each stage in a pair's partials
  int c0[DS_MAX_STAGES + 1];                 // first channel of each stage in alpha / beta
  int n_stages, N, two;
};

constexpr int NMOM = 5;                      // sum x, y, x^2, y^2, xy

__device__ __forceinline__ double bf16_pair_val(uint32_t h, uint32_t l, bool lo_half) {
  return lo_half ? static_cast<double>(bf16_lo(h)) + static_cast<double>(bf16_lo(l))
                 : static_cast<double>(bf16_hi(h)) + static_cast<double>(bf16_hi(l));
}

__device__ __forceinline__ void add_moments(double (&m)[NMOM], double x, double y) {
  m[0] += x;
  m[1] += y;
  m[2] = fma(x, x, m[2]);
  m[3] = fma(y, y, m[3]);
  m[4] = fma(x, y, m[4]);
}

// grid = (blocks of all stages, N).  Stage 0 block = one channel x one chunk (thread = pixel); feature-stage block =
// 64 channels x one chunk (lane = 2 channels, warp = every 8th pixel of the chunk).  Writes the chunk's 5 moments per
// channel to slot (stage, channel, chunk).
__global__ void __launch_bounds__(LP_THREADS) dists_moments_kernel(const __grid_constant__ DistsParams p,
                                                                   double* __restrict__ partial) {
  __shared__ double red[LP_THREADS / 32][DS_GROUP][NMOM];
  const int n = blockIdx.y, blk = blockIdx.x;
  int k = 0;
  while (k + 1 < p.n_stages && blk >= p.blk0[k + 1]) ++k;
  const int local = blk - p.blk0[k], chunks = p.chunks[k], hw = p.hw[k];
  const int grp = local / chunks, j = local - grp * chunks;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int pix0 = j * DS_PIX, pix1 = min(pix0 + DS_PIX, hw);
  double* out = partial + static_cast<int64_t>(n) * p.slot0[p.n_stages] * NMOM;
  if (k == 0) {
    double m[NMOM] = {0.0, 0.0, 0.0, 0.0, 0.0};
    const int64_t plane = (static_cast<int64_t>(n) * 3 + grp) * hw;
    for (int q = pix0 + threadIdx.x; q < pix1; q += LP_THREADS)
      add_moments(m, static_cast<double>(__ldg(p.img0 + plane + q)), static_cast<double>(__ldg(p.img1 + plane + q)));
#pragma unroll
    for (int t = 0; t < NMOM; ++t) {
      m[t] = warp_sum_d(m[t]);
      if (lane == 0) red[warp][0][t] = m[t];
    }
    __syncthreads();
    if (threadIdx.x < NMOM) {
      double s = 0.0;
#pragma unroll
      for (int w = 0; w < LP_THREADS / 32; ++w) s += red[w][0][threadIdx.x];
      out[(static_cast<int64_t>(p.slot0[0]) + grp * chunks + j) * NMOM + threadIdx.x] = s;
    }
    return;
  }
  const bool two = p.two != 0;
  const int C = p.C[k];
  const int c = grp * DS_GROUP + 2 * lane;
  const int64_t img0 = static_cast<int64_t>(n) * hw * C, img1 = static_cast<int64_t>(p.N + n) * hw * C;
  double a[NMOM] = {0.0, 0.0, 0.0, 0.0, 0.0}, b[NMOM] = {0.0, 0.0, 0.0, 0.0, 0.0};
  for (int q = pix0 + warp; q < pix1; q += LP_THREADS / 32) {
    const int64_t o = static_cast<int64_t>(q) * C + c;
    const uint32_t xh = __ldg(reinterpret_cast<const uint32_t*>(p.f0[k] + img0 + o));
    const uint32_t yh = __ldg(reinterpret_cast<const uint32_t*>(p.f0[k] + img1 + o));
    const uint32_t xl = two ? __ldg(reinterpret_cast<const uint32_t*>(p.f1[k] + img0 + o)) : 0u;
    const uint32_t yl = two ? __ldg(reinterpret_cast<const uint32_t*>(p.f1[k] + img1 + o)) : 0u;
    add_moments(a, bf16_pair_val(xh, xl, true), bf16_pair_val(yh, yl, true));
    add_moments(b, bf16_pair_val(xh, xl, false), bf16_pair_val(yh, yl, false));
  }
#pragma unroll
  for (int t = 0; t < NMOM; ++t) red[warp][2 * lane][t] = a[t], red[warp][2 * lane + 1][t] = b[t];
  __syncthreads();
  for (int e = threadIdx.x; e < DS_GROUP * NMOM; e += LP_THREADS) {
    const int cc = e / NMOM, t = e - cc * NMOM;
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < LP_THREADS / 32; ++w) s += red[w][cc][t];
    out[(static_cast<int64_t>(p.slot0[k]) + (grp * DS_GROUP + cc) * chunks + j) * NMOM + t] = s;
  }
}

// One block per image pair: per channel (thread = every 256th channel) the fixed-order sum of its chunk moments, S1
// and S2, weighted by alpha / beta; then the fixed-order sum over the channels.  The weight sum runs through the same
// reduction, so D(x, x) = 1 - w / w = 0 exactly.  __d*_rn keep the compiler from contracting into fma, which would make
// mx^2 + my^2 depend on the operand order.
__global__ void __launch_bounds__(LP_THREADS) dists_finish_kernel(const __grid_constant__ DistsParams p,
                                                                  const double* __restrict__ partial,
                                                                  float* __restrict__ out) {
  __shared__ double red[2][LP_THREADS / 32];
  const int n = blockIdx.x;
  const double* q = partial + static_cast<int64_t>(n) * p.slot0[p.n_stages] * NMOM;
  double acc = 0.0, wsum = 0.0;
  int k = 0;
  for (int c = threadIdx.x; c < p.c0[p.n_stages]; c += LP_THREADS) {
    while (c >= p.c0[k + 1]) ++k;
    const int chunks = p.chunks[k];
    const double* s = q + (static_cast<int64_t>(p.slot0[k]) + (c - p.c0[k]) * chunks) * NMOM;
    double m[NMOM] = {0.0, 0.0, 0.0, 0.0, 0.0};
    for (int j = 0; j < chunks; ++j) {
#pragma unroll
      for (int t = 0; t < NMOM; ++t) m[t] += s[j * NMOM + t];
    }
    const double hw = static_cast<double>(p.hw[k]);
    const double mx = __ddiv_rn(m[0], hw), my = __ddiv_rn(m[1], hw);
    const double exx = __ddiv_rn(m[2], hw), eyy = __ddiv_rn(m[3], hw), exy = __ddiv_rn(m[4], hw);
    const double mxx = __dmul_rn(mx, mx), myy = __dmul_rn(my, my), mxy = __dmul_rn(mx, my);
    const double vx = __dsub_rn(exx, mxx), vy = __dsub_rn(eyy, myy), cov = __dsub_rn(exy, mxy);
    const double s1 = __ddiv_rn(__dadd_rn(__dmul_rn(2.0, mxy), DS_C1), __dadd_rn(__dadd_rn(mxx, myy), DS_C1));
    const double s2 = __ddiv_rn(__dadd_rn(__dmul_rn(2.0, cov), DS_C2), __dadd_rn(__dadd_rn(vx, vy), DS_C2));
    const double al = static_cast<double>(__ldg(p.alpha + c)), be = static_cast<double>(__ldg(p.beta + c));
    acc = __dadd_rn(acc, __dadd_rn(__dmul_rn(al, s1), __dmul_rn(be, s2)));
    wsum = __dadd_rn(wsum, __dadd_rn(al, be));
  }
  acc = warp_sum_d(acc);
  wsum = warp_sum_d(wsum);
  const int warp = threadIdx.x >> 5;
  if ((threadIdx.x & 31) == 0) red[0][warp] = acc, red[1][warp] = wsum;
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0.0, w = 0.0;
#pragma unroll
    for (int i = 0; i < LP_THREADS / 32; ++i) a += red[0][i], w += red[1][i];
    out[n] = static_cast<float>(__dsub_rn(1.0, __ddiv_rn(a, w)));
  }
}

int dists_params(int H, int W, const b200dn_dists_stage* stages, int n_stages, int N, int prec, DistsParams& p) {
  B200DN_CHECK_ARG(stages && n_stages >= 1 && n_stages < DS_MAX_STAGES, "dists_head: 1..%d feature stages",
                   DS_MAX_STAGES - 1);
  B200DN_CHECK_ARG(N >= 1 && N <= 65535, "dists_head: 1..65535 image pairs");
  B200DN_CHECK_ARG(H > 0 && W > 0 && static_cast<int64_t>(H) * W < (1 << 30), "dists_head: bad image size %d x %d", H, W);
  B200DN_CHECK_ARG(bf16_prec(prec), "dists_head: prec %d: only the bf16-stored precisions are supported", prec);
  memset(&p, 0, sizeof(p));
  p.n_stages = n_stages + 1, p.N = N, p.two = two_planes(prec) ? 1 : 0;
  int64_t blocks = 0, slots = 0, chans = 0;
  for (int k = 0; k <= n_stages; ++k) {
    int h = H, w = W, c = 3;
    if (k > 0) {
      const b200dn_dists_stage& s = stages[k - 1];
      B200DN_CHECK_ARG(s.feat[0] && (!p.two || s.feat[1]), "dists_head: stage %d: null pointer", k);
      B200DN_CHECK_ARG(((reinterpret_cast<uintptr_t>(s.feat[0]) | reinterpret_cast<uintptr_t>(s.feat[1])) & 15) == 0,
                       "dists_head: stage %d: feature planes must be 16-byte aligned", k);
      B200DN_CHECK_ARG(s.H > 0 && s.W > 0 && static_cast<int64_t>(s.H) * s.W < (1 << 30) && s.C > 0 &&
                           s.C % DS_GROUP == 0,
                       "dists_head: stage %d: H, W > 0 and C a multiple of %d (got %d x %d x %d)", k, DS_GROUP, s.H,
                       s.W, s.C);
      p.f0[k] = static_cast<const uint16_t*>(s.feat[0]);
      p.f1[k] = static_cast<const uint16_t*>(s.feat[1]);
      h = s.H, w = s.W, c = s.C;
    }
    p.hw[k] = h * w;
    p.C[k] = c;
    p.chunks[k] = static_cast<int>(cdiv64(static_cast<int64_t>(h) * w, DS_PIX));
    p.blk0[k] = static_cast<int>(blocks);
    p.slot0[k] = static_cast<int>(slots);
    p.c0[k] = static_cast<int>(chans);
    blocks += static_cast<int64_t>(k == 0 ? c : c / DS_GROUP) * p.chunks[k];
    slots += static_cast<int64_t>(c) * p.chunks[k];
    chans += c;
    B200DN_CHECK_ARG(blocks < (1 << 30) && slots < (1 << 26), "dists_head: too many pixels");
  }
  p.blk0[p.n_stages] = static_cast<int>(blocks);
  p.slot0[p.n_stages] = static_cast<int>(slots);
  p.c0[p.n_stages] = static_cast<int>(chans);
  return 0;
}

}  // namespace
}  // namespace b200dn

extern "C" int b200dn_l2pool3x3s2(const void* in_hi, const void* in_lo, int B, int H, int W, int C,
                                  const float* filter, int prec, void* out0, void* out1, void* stream) {
  using namespace b200dn;
  B200DN_CHECK_ARG(in_hi && out0 && filter, "l2pool3x3s2: null pointer");
  B200DN_CHECK_ARG(bf16_prec(prec), "l2pool3x3s2: prec %d: only the bf16-stored precisions are supported", prec);
  B200DN_CHECK_ARG(!two_planes(prec) || (in_lo && out1), "l2pool3x3s2: prec %d needs the lo planes", prec);
  B200DN_CHECK_ARG(B > 0 && H >= 1 && W >= 1 && C > 0 && C % 8 == 0,
                   "l2pool3x3s2: needs H, W >= 1 and C a multiple of 8 (got %d x %d x %d)", H, W, C);
  B200DN_CHECK_ARG(((reinterpret_cast<uintptr_t>(in_hi) | reinterpret_cast<uintptr_t>(in_lo) |
                     reinterpret_cast<uintptr_t>(out0) | reinterpret_cast<uintptr_t>(out1)) & 15) == 0,
                   "l2pool3x3s2: planes must be 16-byte aligned");
  if (int rc = require_sm100()) return rc;
  const int Ho = (H - 1) / 2 + 1, Wo = (W - 1) / 2 + 1;
  const int grid = lp_grid(static_cast<int64_t>(B) * Ho * Wo * (C / 8));
  if (grid <= 0) return B200DN_E_CUDA;
  l2pool_kernel<<<grid, LP_THREADS, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const uint16_t*>(in_hi), static_cast<const uint16_t*>(in_lo), B, H, W, C, filter, Ho, Wo,
      two_planes(prec) ? 1 : 0, static_cast<uint16_t*>(out0), static_cast<uint16_t*>(out1));
  B200DN_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int64_t b200dn_dists_head_workspace_bytes(int H, int W, const b200dn_dists_stage* stages, int n_stages,
                                                     int N) {
  b200dn::DistsParams p;
  if (b200dn::dists_params(H, W, stages, n_stages, N, B200DN_PREC_BF16, p)) return 0;
  return static_cast<int64_t>(N) * p.slot0[p.n_stages] * b200dn::NMOM * static_cast<int64_t>(sizeof(double));
}

extern "C" int b200dn_dists_head(const float* in0, const float* in1, int H, int W, const b200dn_dists_stage* stages,
                                 int n_stages, int N, const float* alpha, const float* beta, int prec, float* out,
                                 void* workspace, int64_t workspace_bytes, void* stream) {
  using namespace b200dn;
  DistsParams p;
  if (int rc = dists_params(H, W, stages, n_stages, N, prec, p)) return rc;
  B200DN_CHECK_ARG(in0 && in1 && alpha && beta && out, "dists_head: null pointer");
  B200DN_CHECK_ARG(workspace && (reinterpret_cast<uintptr_t>(workspace) & 7) == 0 &&
                       workspace_bytes >= static_cast<int64_t>(N) * p.slot0[p.n_stages] * NMOM *
                                              static_cast<int64_t>(sizeof(double)),
                   "dists_head: workspace of b200dn_dists_head_workspace_bytes() bytes (8-byte aligned) required");
  if (int rc = require_sm100()) return rc;
  p.img0 = in0, p.img1 = in1, p.alpha = alpha, p.beta = beta;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  double* partial = static_cast<double*>(workspace);
  dists_moments_kernel<<<dim3(static_cast<unsigned>(p.blk0[p.n_stages]), static_cast<unsigned>(N)), LP_THREADS, 0, s>>>(
      p, partial);
  B200DN_CUDA(cudaGetLastError());
  dists_finish_kernel<<<static_cast<unsigned>(N), LP_THREADS, 0, s>>>(p, partial, out);
  B200DN_CUDA(cudaGetLastError());
  return 0;
}

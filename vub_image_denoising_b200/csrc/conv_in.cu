// conv_in.cu — InputBlock.conv_1 + actv_1 (UNet/RDUNet_model.py:71-81) fused with the module-boundary
// ingest: reads the caller's fp32 NCHW image (and, for RDUNet_T, the broadcast timestep plane that the
// reference concatenates at diffusion_denoising/Unet/Unet_model.py:135-136), writes NHWC 16-bit planes.
// K = 27 or 36 is far too small for the tensor pipe and the layer is bandwidth-bound (AI ~ 26 FLOP/B),
// so this runs on CUDA cores in fp32.
#include "igemm_common.cuh"

#include <stdlib.h>

namespace b200dn {

namespace {

constexpr int PX = 32;     // pixels along W per block (one warp = 32 consecutive pixels: coalesced NCHW reads)
constexpr int ROWS = 8;    // warps per block; each thread owns TWO vertically adjacent pixels per pass
constexpr int PASSES = 4;  // a block covers PX x (2 * ROWS * PASSES) pixels, so the weights are staged once per 2048 px

__device__ __forceinline__ uint32_t pack_f16x2_sat(float lo, float hi) {   // saturates at +-65504 like the igemm epilogue
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ uint32_t sat_track(uint32_t m, uint32_t h) {
  uint32_t r;
  asm("{\n\t.reg .b32 a;\n\tabs.f16x2 a, %2;\n\tmax.NaN.f16x2 %0, %1, a;\n\t}" : "=r"(r) : "r"(m), "r"(h));
  return r;
}

template <bool kBf16>
__device__ __forceinline__ void store_group(const float (&acc)[8], const float* b_s, const float* s_s, int g,
                                            uint16_t* o0, uint16_t* o1, uint32_t& satm) {
  uint32_t hi[4], lo[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    float a = acc[2 * j] + b_s[g * 8 + 2 * j];
    float c = acc[2 * j + 1] + b_s[g * 8 + 2 * j + 1];
    a = a > 0.f ? a : a * s_s[g * 8 + 2 * j];
    c = c > 0.f ? c : c * s_s[g * 8 + 2 * j + 1];
    if (kBf16) {
      hi[j] = pack_bf16x2(a, c);
      lo[j] = pack_bf16x2(a - bf16_lo(hi[j]), c - bf16_hi(hi[j]));
    } else {
      hi[j] = pack_f16x2_sat(a, c);
      lo[j] = pack_f16x2_sat(a - f16_lo(hi[j]), c - f16_hi(hi[j]));
      satm = sat_track(satm, hi[j]);
    }
  }
  *reinterpret_cast<uint4*>(o0 + g * 8) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
  if (o1 != nullptr) *reinterpret_cast<uint4*>(o1 + g * 8) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
}

// One thread = two vertically adjacent pixels, all output channels in groups of 8.  The weights are broadcast from
// shared memory (2 x LDS.128 per k and group); sharing them between two pixels halves the shared-memory reads per FMA
// (the one-pixel version issued one LDS.128 per 4 FFMA and ran at a third of the FP32 rate), and the two pixels share
// 8 of their 12 input rows x columns.
// CIMG = channels of the image (3 RGB, 1 grayscale); HAS_T = the RDUNet_T timestep plane as an extra input channel
template <int CIMG, bool HAS_T>
__global__ void __launch_bounds__(PX * ROWS) conv_in_kernel(const float* __restrict__ x, int Bx,
                                                            const float* __restrict__ t, int64_t t_sb, int64_t t_sh,
                                                            int64_t t_sw, int H, int W, int cout,
                                                            const float* __restrict__ w, const float* __restrict__ bias,
                                                            const float* __restrict__ slope, int prec,
                                                            uint16_t* __restrict__ out0, uint16_t* __restrict__ out1,
                                                            int out_ctot, int* __restrict__ sat_flag) {
  constexpr int CIN = CIMG + (HAS_T ? 1 : 0);
  extern __shared__ float w_s[];  // [CIN*9][cout], then bias[cout], slope[cout]
  constexpr int K = CIN * 9;
  float* b_s = w_s + K * cout;
  float* s_s = b_s + cout;
  const int tid = threadIdx.y * PX + threadIdx.x;
  for (int i = tid; i < K * cout; i += PX * ROWS) {
    const int o = i / K, k = i - o * K;  // w is [o][ci][ky][kx] = [o][k]
    w_s[k * cout + o] = w[i];
  }
  for (int i = tid; i < cout; i += PX * ROWS) {
    b_s[i] = bias[i];
    s_s[i] = slope[i];
  }
  __syncthreads();

  const int b = blockIdx.z;
  const int xx = blockIdx.x * PX + threadIdx.x;
  const int64_t hw = static_cast<int64_t>(H) * W;
  const float* xb = x + static_cast<int64_t>(b % Bx) * CIMG * hw;
  const bool is_bf16 = (prec != B200DN_PREC_FP16) && (prec != B200DN_PREC_FP16X2);
  if (xx >= W) return;
  uint32_t satm = 0;

  for (int pass = 0; pass < PASSES; ++pass) {
    const int y = ((blockIdx.y * PASSES + pass) * ROWS + threadIdx.y) * 2;   // rows y and y + 1
    if (y >= H) break;
    const bool two = (y + 1) < H;
    float v[CIN][4][3];   // input rows y-1 .. y+2, columns xx-1 .. xx+1
#pragma unroll
    for (int r = 0; r < 4; ++r) {
#pragma unroll
      for (int kx = 0; kx < 3; ++kx) {
        const int yy = y + r - 1, xc = xx + kx - 1;
        const bool in = (yy >= 0) && (yy < H) && (xc >= 0) && (xc < W);
        const int64_t sp = static_cast<int64_t>(yy) * W + xc;
#pragma unroll
        for (int ci = 0; ci < CIMG; ++ci) v[ci][r][kx] = in ? __ldg(xb + ci * hw + sp) : 0.f;
        if (HAS_T) v[CIMG][r][kx] = in ? __ldg(t + b * t_sb + yy * t_sh + xc * t_sw) : 0.f;
      }
    }
    const int64_t pix = (static_cast<int64_t>(b) * H + y) * W + xx;
    uint16_t* o0 = out0 + pix * out_ctot;
    uint16_t* o1 = out1 ? out1 + pix * out_ctot : nullptr;
    const int64_t row = static_cast<int64_t>(W) * out_ctot;
    for (int g = 0; g * 8 < cout; ++g) {
      // packed fp32 FMAs (FFMA2: two IEEE fmas per instruction, same bits as fmaf) — the kernel is FP32-issue-bound
      float2 p0[4], p1[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) p0[j] = p1[j] = make_float2(0.f, 0.f);
#pragma unroll
      for (int ci = 0; ci < CIN; ++ci) {
#pragma unroll
        for (int ky = 0; ky < 3; ++ky) {
#pragma unroll
          for (int kx = 0; kx < 3; ++kx) {
            const int k = ci * 9 + ky * 3 + kx;
            const float4 w0 = *reinterpret_cast<const float4*>(w_s + k * cout + g * 8);
            const float4 w1 = *reinterpret_cast<const float4*>(w_s + k * cout + g * 8 + 4);
            const float2 a = make_float2(v[ci][ky][kx], v[ci][ky][kx]);
            const float2 c = make_float2(v[ci][ky + 1][kx], v[ci][ky + 1][kx]);
            const float2 wa = make_float2(w0.x, w0.y), wb = make_float2(w0.z, w0.w);
            const float2 wc = make_float2(w1.x, w1.y), wd = make_float2(w1.z, w1.w);
            p0[0] = __ffma2_rn(a, wa, p0[0]);
            p0[1] = __ffma2_rn(a, wb, p0[1]);
            p0[2] = __ffma2_rn(a, wc, p0[2]);
            p0[3] = __ffma2_rn(a, wd, p0[3]);
            p1[0] = __ffma2_rn(c, wa, p1[0]);
            p1[1] = __ffma2_rn(c, wb, p1[1]);
            p1[2] = __ffma2_rn(c, wc, p1[2]);
            p1[3] = __ffma2_rn(c, wd, p1[3]);
          }
        }
      }
      float acc0[8], acc1[8];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        acc0[2 * j] = p0[j].x, acc0[2 * j + 1] = p0[j].y;
        acc1[2 * j] = p1[j].x, acc1[2 * j + 1] = p1[j].y;
      }
      if (is_bf16) {
        store_group<true>(acc0, b_s, s_s, g, o0, o1, satm);
        if (two) store_group<true>(acc1, b_s, s_s, g, o0 + row, o1 ? o1 + row : nullptr, satm);
      } else {
        store_group<false>(acc0, b_s, s_s, g, o0, o1, satm);
        if (two) store_group<false>(acc1, b_s, s_s, g, o0 + row, o1 ? o1 + row : nullptr, satm);
      }
    }
  }
  if (sat_flag != nullptr && (((satm & 0x7fffu) >= 0x7bffu) || ((satm >> 16) >= 0x7bffu))) atomicOr(sat_flag, 1);
}

}  // namespace
}  // namespace b200dn

namespace b200dn {
// ---------------------------------------------------------------------------------------------------------------
// Tensor-core ingest (single-plane bf16 / fp16 modes).  The CUDA-core kernel above is fp32-FMA bound: 2.4 GFMA for
// RDUNet_T(32) at B = 32 = 145 us = 3.3 % of a sampler step, 0.83 ms of the RDUNet(128) step (ncu launch lists,
// profiles/r02_*_launches.csv).  Here the K = 27 / 36 (ci, ky, kx) patch of every pixel is gathered once into a
// K-major 128-byte-swizzled A tile in shared memory as TWO 16-bit planes (hi + lo: the fp32 image keeps 22 of its 24
// bits in fp16 and 16 in bf16, twice the precision of the 16-bit output or more), the conv weights sit resident as one 16-bit plane (the same rounding every
// other layer's weights get) and the layer is 2 x ceil(K / 16) tcgen05.mma per 128 pixels.
// Warp roles (416 threads): 0-3 and 9-12 = two epilogue groups (one half of the accumulator columns each: with one
// group the 128-channel ingest ran 2 % slower), 4-7 and 13-16 = two gather groups (thread = pixel of an 8 x 16 tile; group
// g fills A stage g for the CTA's even / odd tiles — the gather, ~300 instructions per pixel behind its image loads,
// is what paces a tile), 8 = TMEM allocator + MMA issuer.
namespace ingest_tc {
using namespace igemm;
constexpr int TW_ = SLAB_TILE_W, TH_ = SLAB_TILE_H;           // 8 x 16 pixels = 128 accumulator rows
constexpr int A_PLANE_BYTES = 128 * 128;                      // [128 px][64 k] 16-bit, 128-byte swizzled rows
constexpr int STAGES = 2;
constexpr int MAX_COUT = 256;
constexpr uint32_t OFF_W = 0;                                  // [cout_pad][64 k]: up to 32 KB
constexpr uint32_t OFF_A = MAX_COUT * 128;                     // STAGES x {hi, lo}
constexpr uint32_t OFF_BAR = OFF_A + STAGES * 2 * A_PLANE_BYTES;
constexpr uint32_t OFF_EPI = OFF_BAR + 128;                    // bias[256], slope[256]
// twin mode: per border class (first / inner / last row x column) and output channel, the sum of the 16-bit-rounded
// t-plane weights over the taps that fall inside the image
constexpr uint32_t OFF_TS = OFF_EPI + 2 * MAX_COUT * 4;
constexpr uint32_t SMEM = 1024 + OFF_TS + 9 * MAX_COUT * 4;
constexpr uint32_t B_AFULL = 0, B_AEMPTY = 16, B_TFULL = 32, B_TEMPTY = 48, B_TMEMPTR = 64;
constexpr int THREADS = 544;   // 17 warps: 0-3 / 9-12 epilogue groups (column halves), 4-7 / 13-16 gather groups, 8 issuer

// kTwin (the sampler's call: B = 2 * Bx network images read the SAME Bx input images and differ only in a per-image
// timestep, diffusion_RDUnet.py:43-47): the conv is linear, so conv_1([x, t]) = W_rgb * x + t * S with S the sum of the t-plane
// weights over the in-image taps — a function of the pixel's border class only.  The image part is gathered and multiplied
// ONCE per input image (K = 27) and the epilogue writes both network images, prelu(acc + b + t_a S) and prelu(acc + b + t_b S):
// half the gather, which is what paces this kernel.
template <int CIMG, bool HAS_T, bool kBf16, bool kTwin>
__global__ void __launch_bounds__(THREADS, 1) conv_in_tc_kernel(const float* __restrict__ x, int Bx, const float* __restrict__ t,
                                                                int64_t t_sb, int64_t t_sh, int64_t t_sw, int B, int H, int W,
                                                                int cout, const float* __restrict__ w,
                                                                const float* __restrict__ bias, const float* __restrict__ slope,
                                                                uint16_t* __restrict__ out0, int out_ctot, int* sat_flag) {
  static_assert(!kTwin || HAS_T, "twin mode is the timestep network's");
  constexpr int CIN = CIMG + (HAS_T ? 1 : 0);
  constexpr int KW = CIN * 9;                                  // row length of w
  constexpr int K = (kTwin ? CIMG : CIN) * 9;                  // K of the MMA (twin: the t plane is added in the epilogue)
  constexpr bool GATHER_T = HAS_T && !kTwin;
  constexpr int NK16 = (K + 15) / 16;                          // 2 (K = 9, 18, 27) or 3 (K = 36)
  constexpr int NCHUNK = NK16 * 2;                             // 16-byte chunks (8 k) written per row and plane
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_u32 = smem_u32(smem_raw);
  const uint32_t sb = (raw_u32 + 1023u) & ~1023u;
  uint8_t* sg = smem_raw + (sb - raw_u32);
  const uint32_t bars = sb + OFF_BAR;
  uint32_t* tmem_ptr_s = reinterpret_cast<uint32_t*>(sg + OFF_BAR + B_TMEMPTR);
  float* epi_bias = reinterpret_cast<float*>(sg + OFF_EPI);
  float* epi_slope = epi_bias + MAX_COUT;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int block_n = (cout + 15) & ~15;
  uint32_t tmem_cols = 32;
  while (tmem_cols < static_cast<uint32_t>(STAGES * block_n)) tmem_cols <<= 1;
  const int n_groups = (block_n % 32 == 0) ? 2 : 1;           // epilogue groups that have columns to drain

  if (warp == 8) {
    if (lane == 0) {
      for (int s = 0; s < STAGES; ++s) {
        mbar_init(bars + B_AFULL + s * 8, 4);     // one arrive per gather warp
        mbar_init(bars + B_AEMPTY + s * 8, 1);    // tcgen05.commit
        mbar_init(bars + B_TFULL + s * 8, 1);     // tcgen05.commit
        mbar_init(bars + B_TEMPTY + s * 8, 4 * n_groups);    // one arrive per active epilogue warp
      }
      mbar_fence_init();
    }
    __syncwarp();
    tmem_alloc(smem_u32(tmem_ptr_s), tmem_cols);
    tmem_relinquish();
  }
  // resident weights: [n][k = ci*9 + ky*3 + kx] 16-bit, K-major 128-byte swizzled rows, zero padded (generic-proxy stores)
  for (int i = threadIdx.x; i < block_n * 8; i += THREADS) {
    const int n = i >> 3, chunk = i & 7;
    uint32_t v[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int k0 = chunk * 8 + 2 * q;
      const float a = (n < cout && k0 < K) ? __ldg(w + n * KW + k0) : 0.f;
      const float c = (n < cout && k0 + 1 < K) ? __ldg(w + n * KW + k0 + 1) : 0.f;
      v[q] = kBf16 ? pack_bf16x2(a, c) : pack_f16x2(a, c);
    }
    *reinterpret_cast<uint4*>(sg + OFF_W + n * 128 + ((chunk ^ (n & 7)) << 4)) = make_uint4(v[0], v[1], v[2], v[3]);
  }
  for (int i = threadIdx.x; i < block_n; i += THREADS) {
    epi_bias[i] = i < cout ? __ldg(bias + i) : 0.f;
    epi_slope[i] = i < cout ? __ldg(slope + i) : 1.f;
  }
  float* t_sum = reinterpret_cast<float*>(sg + OFF_TS);         // [class = 3 * ycls + xcls][MAX_COUT]
  if (kTwin) {
    for (int i = threadIdx.x; i < 9 * block_n; i += THREADS) {
      const int cls = i / block_n, n = i - cls * block_n;
      const int ycls = cls / 3, xcls = cls - ycls * 3;          // 0 first row / column, 1 inner, 2 last
      float sum = 0.f;
      if (n < cout) {
        for (int ky = (ycls == 0 ? 1 : 0); ky < (ycls == 2 ? 2 : 3); ++ky)
          for (int kx = (xcls == 0 ? 1 : 0); kx < (xcls == 2 ? 2 : 3); ++kx) {
            const float wv = __ldg(w + n * KW + CIMG * 9 + ky * 3 + kx);
            sum += kBf16 ? bf16_lo(pack_bf16x2(wv, 0.f)) : f16_lo(pack_f16x2(wv, 0.f));   // the 16-bit weight the MMA would use
          }
      }
      t_sum[cls * MAX_COUT + n] = sum;
    }
  }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_s;
  griddep_launch_dependents();

  const int tiles_x = (W + TW_ - 1) / TW_, tiles_y = (H + TH_ - 1) / TH_;
  const int num_tiles = (kTwin ? Bx : B) * tiles_x * tiles_y, grid = gridDim.x;     // twin: one tile per INPUT image tile
  const int64_t hw = static_cast<int64_t>(H) * W;

  if ((warp >= 4 && warp < 8) || warp >= 13) {
    // ===================================================== gather: thread = pixel, im2col row -> A tile (hi, lo planes)
    griddep_wait();      // x may be the previous kernel's output (the sampler's x_t)
    const int gg = warp >= 13 ? 1 : 0;                         // gather group = A stage = parity of the CTA-local tile index
    const int pxl = ((warp - 4) & 3) * 32 + lane;              // warps 4-7 -> 0..3, warps 13-16 -> (9..12) & 3 = 1,2,3,0
    const int th = pxl >> 3, tw = pxl & 7;
    const uint32_t row_off = static_cast<uint32_t>(pxl) * 128u, swz = static_cast<uint32_t>(pxl & 7);
    TileWalker wk;
    wk.init(blockIdx.x + gg * grid, 2 * grid, 1, tiles_x, tiles_y);
    int it = gg;
    for (int tile = blockIdx.x + gg * grid; tile < num_tiles; tile += 2 * grid, wk.next(), it += 2) {
      const int st = gg;
      const uint32_t ph = static_cast<uint32_t>((it >> 1) & 1);
      const int b = wk.b, y = wk.ty * TH_ + th, xx = wk.tx * TW_ + tw;
      const float* xb = x + static_cast<int64_t>(b % Bx) * CIMG * hw;
      float v[NCHUNK * 8];
#pragma unroll
      for (int k = K; k < NCHUNK * 8; ++k) v[k] = 0.f;
#pragma unroll
      for (int ky = 0; ky < 3; ++ky) {
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
          const int yy = y + ky - 1, xc = xx + kx - 1;
          const bool in = (yy >= 0) && (yy < H) && (xc >= 0) && (xc < W);
          const int64_t sp = static_cast<int64_t>(yy) * W + xc;
#pragma unroll
          for (int ci = 0; ci < CIMG; ++ci) v[ci * 9 + ky * 3 + kx] = in ? __ldg(xb + ci * hw + sp) : 0.f;
          if (GATHER_T) v[CIMG * 9 + ky * 3 + kx] = in ? __ldg(t + b * t_sb + yy * t_sh + xc * t_sw) : 0.f;
        }
      }
      mbar_wait(bars + B_AEMPTY + st * 8, ph ^ 1u);       // the MMAs that read this stage have retired
      uint8_t* a_hi = sg + OFF_A + (st * 2) * A_PLANE_BYTES + row_off;
      uint8_t* a_lo = a_hi + A_PLANE_BYTES;
#pragma unroll
      for (int c = 0; c < NCHUNK; ++c) {
        uint32_t hi[4], lo[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float a = v[c * 8 + 2 * q], d = v[c * 8 + 2 * q + 1];
          hi[q] = kBf16 ? pack_bf16x2(a, d) : pack_f16x2(a, d);
          const float ra = a - (kBf16 ? bf16_lo(hi[q]) : f16_lo(hi[q])), rd = d - (kBf16 ? bf16_hi(hi[q]) : f16_hi(hi[q]));
          lo[q] = kBf16 ? pack_bf16x2(ra, rd) : pack_f16x2(ra, rd);
        }
        const uint32_t off = (static_cast<uint32_t>(c) ^ swz) << 4;
        *reinterpret_cast<uint4*>(a_hi + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        *reinterpret_cast<uint4*>(a_lo + off) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(bars + B_AFULL + st * 8);
    }
  } else if (warp == 8) {
    // ===================================================== MMA issuer: D = A_lo W + A_hi W, 2 x NK16 UMMAs per tile
    const uint32_t idesc = make_idesc_f16(kBf16 ? 1u : 0u, static_cast<uint32_t>(block_n));
    const uint64_t bdesc = make_sw128_desc(sb + OFF_W, 1024);
    int it = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += grid, ++it) {
      const int st = it & 1;
      const uint32_t ph = static_cast<uint32_t>((it >> 1) & 1);
      mbar_wait(bars + B_TEMPTY + st * 8, ph ^ 1u);       // accumulator stage drained
      mbar_wait(bars + B_AFULL + st * 8, ph);
      tc_fence_after();
      if (elect_one()) {
        const uint32_t d = tmem_base + static_cast<uint32_t>(st * block_n);
        const uint64_t a_hi = make_sw128_desc(sb + OFF_A + (st * 2) * A_PLANE_BYTES, 1024);
        const uint64_t a_lo = make_sw128_desc(sb + OFF_A + (st * 2 + 1) * A_PLANE_BYTES, 1024);
#pragma unroll
        for (int k = 0; k < NK16; ++k) umma_f16(d, a_lo + 2 * k, bdesc + 2 * k, idesc, k == 0 ? 0u : 1u);   // small term first
#pragma unroll
        for (int k = 0; k < NK16; ++k) umma_f16(d, a_hi + 2 * k, bdesc + 2 * k, idesc, 1u);
        umma_commit(bars + B_AEMPTY + st * 8);
        umma_commit(bars + B_TFULL + st * 8);
      }
      __syncwarp();
    }
  } else if (warp < 4 || (warp >= 9 && n_groups == 2)) {
    // ===================================================== epilogue: bias + PReLU -> 16-bit NHWC channels [0, cout)
    griddep_wait();      // WAR: the previous kernel may still read the buffer this layer writes
    const int grp = warp >= 9 ? 1 : 0;
    const int we = warp & 3;                                    // TMEM lane quarter this warp may read
    const int ncols = block_n / n_groups, col0 = grp * ncols;
    const int row = we * 32 + lane;
    const int th = row >> 3, tw = row & 7;
    EpiArgs ea;
    ea.out0 = out0, ea.out1 = nullptr, ea.res0 = nullptr, ea.res1 = nullptr;
    ea.out_ctot = out_ctot, ea.out_coff = 0, ea.res_ctot = 0, ea.cout = cout;
    ea.out_kind = B200DN_OUT_NHWC16, ea.is_bf16 = kBf16 ? 1 : 0;
    ea.out_nchw = nullptr, ea.res_nchw = nullptr, ea.res_bmod = 1, ea.H = H, ea.W = W;
    ea.sat_flag = kBf16 ? nullptr : sat_flag;
    uint32_t satm = 0;
    TileWalker wk;
    wk.init(blockIdx.x, grid, 1, tiles_x, tiles_y);
    int it = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += grid, wk.next(), ++it) {
      const int st = it & 1;
      const uint32_t ph = static_cast<uint32_t>((it >> 1) & 1);
      const int b = wk.b, y = wk.ty * TH_ + th, xx = wk.tx * TW_ + tw;
      const bool valid = (y < H) && (xx < W);
      const int64_t pix = (static_cast<int64_t>(b) * H + y) * W + xx;
      mbar_wait(bars + B_TFULL + st * 8, ph);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(we * 32) << 16) + static_cast<uint32_t>(st * block_n + col0);
      if (!kTwin) {
        epilogue_subtile(ea, taddr, ncols, epi_bias + col0, epi_slope + col0, valid, b, y, xx, pix, pix, col0,
                         bars + B_TEMPTY + st * 8, satm);
        continue;
      }
      // twin: both network images of this input pixel from one accumulator
      float tj[2] = {0.f, 0.f};
      if (valid) tj[0] = __ldg(t + b * t_sb), tj[1] = __ldg(t + (b + Bx) * t_sb);
      const int cls = (y == 0 ? 0 : y == H - 1 ? 2 : 1) * 3 + (xx == 0 ? 0 : xx == W - 1 ? 2 : 1);
      const float* ts = t_sum + cls * MAX_COUT + col0;
      for (int c0 = 0; c0 < ncols; c0 += 16) {
        uint32_t r[16];
        tmem_ld16(taddr + c0, r);
        tmem_ld_wait();
        if (c0 + 16 >= ncols) {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(bars + B_TEMPTY + st * 8);
        }
        if (!valid) continue;
        // bias / slopes: broadcast 128-bit loads; S: one 128-bit load per lane and 4 columns (its border class's row)
        float base[16], sv[16], sl[16];
        const float4* b4 = reinterpret_cast<const float4*>(epi_bias + col0 + c0);
        const float4* s4 = reinterpret_cast<const float4*>(epi_slope + col0 + c0);
        const float4* t4 = reinterpret_cast<const float4*>(ts + c0);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float4 bb = b4[q], ss = s4[q], tt = t4[q];
          base[4 * q] = __uint_as_float(r[4 * q]) + bb.x, base[4 * q + 1] = __uint_as_float(r[4 * q + 1]) + bb.y;
          base[4 * q + 2] = __uint_as_float(r[4 * q + 2]) + bb.z, base[4 * q + 3] = __uint_as_float(r[4 * q + 3]) + bb.w;
          sl[4 * q] = ss.x, sl[4 * q + 1] = ss.y, sl[4 * q + 2] = ss.z, sl[4 * q + 3] = ss.w;
          sv[4 * q] = tt.x, sv[4 * q + 1] = tt.y, sv[4 * q + 2] = tt.z, sv[4 * q + 3] = tt.w;
        }
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          uint32_t h[8];
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            float a0 = base[2 * q] + tj[j] * sv[2 * q], a1 = base[2 * q + 1] + tj[j] * sv[2 * q + 1];
            a0 = a0 > 0.f ? a0 : a0 * sl[2 * q];
            a1 = a1 > 0.f ? a1 : a1 * sl[2 * q + 1];
            h[q] = pack2<kBf16>(a0, a1);
          }
          if (!kBf16 && ea.sat_flag != nullptr) {
#pragma unroll
            for (int q = 0; q < 8; ++q) satm = igemm::sat_track(satm, h[q]);
          }
          const int64_t pj = pix + static_cast<int64_t>(j) * Bx * hw;
          uint4* dst = reinterpret_cast<uint4*>(out0 + pj * out_ctot + col0 + c0);
          dst[0] = make_uint4(h[0], h[1], h[2], h[3]);
          if (col0 + c0 + 8 < cout) dst[1] = make_uint4(h[4], h[5], h[6], h[7]);
        }
      }
    }
    sat_report(ea.sat_flag, satm);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 8) {
    tc_fence_after();
    tmem_dealloc(tmem_base, tmem_cols);
  }
}

template <int CIMG, bool HAS_T, bool kTwin>
int launch(int grid, cudaStream_t s, const float* x, int Bx, const float* t, int64_t t_sb, int64_t t_sh, int64_t t_sw, int B,
           int H, int W, int cout, const float* w, const float* bias, const float* slope, bool bf16, uint16_t* o0, int out_ctot,
           int* sat_flag) {
  static const void* const kernels[2] = {reinterpret_cast<const void*>(conv_in_tc_kernel<CIMG, HAS_T, false, kTwin>),
                                         reinterpret_cast<const void*>(conv_in_tc_kernel<CIMG, HAS_T, true, kTwin>)};
  static SmemOptIn opt_in;
  if (int rc = ensure_max_dyn_smem(opt_in, kernels, 2, SMEM, "cudaFuncSetAttribute(conv_in_tc_kernel, smem)")) return rc;
  if (bf16)
    conv_in_tc_kernel<CIMG, HAS_T, true, kTwin><<<grid, THREADS, SMEM, s>>>(x, Bx, t, t_sb, t_sh, t_sw, B, H, W, cout, w, bias,
                                                                             slope, o0, out_ctot, sat_flag);
  else
    conv_in_tc_kernel<CIMG, HAS_T, false, kTwin><<<grid, THREADS, SMEM, s>>>(x, Bx, t, t_sb, t_sh, t_sw, B, H, W, cout, w, bias,
                                                                              slope, o0, out_ctot, sat_flag);
  B200DN_CUDA(cudaGetLastError());
  return 0;
}

// B200DN_CONV_IN_TWIN=0: the sampler's 2B batch gathers every input image twice (once per timestep) as a general batch
bool twin_enabled() {
  const char* e = getenv("B200DN_CONV_IN_TWIN");
  return e ? atoi(e) != 0 : true;
}

bool enabled() {
  static int on = [] {
    const char* e = getenv("B200DN_CONV_IN_TC");
    return e ? atoi(e) : 1;
  }();
  return on != 0;
}
}  // namespace ingest_tc

namespace {
template <int CIMG, bool HAS_T>
int launch_conv_in(dim3 grid, dim3 block, size_t smem, cudaStream_t s, const float* x, int Bx, const float* t, int64_t t_sb,
                   int64_t t_sh, int64_t t_sw, int H, int W, int cout, const float* w, const float* bias, const float* slope,
                   int prec, uint16_t* o0, uint16_t* o1, int out_ctot, int* sat_flag) {
  if (smem > 48 * 1024)
    B200DN_CUDA(cudaFuncSetAttribute(conv_in_kernel<CIMG, HAS_T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  conv_in_kernel<CIMG, HAS_T><<<grid, block, smem, s>>>(x, Bx, t, t_sb, t_sh, t_sw, H, W, cout, w, bias, slope, prec, o0, o1,
                                                         out_ctot, sat_flag);
  B200DN_CUDA(cudaGetLastError());
  return 0;
}
}  // namespace
}  // namespace b200dn

extern "C" int b200dn_conv_in(const float* x, int Bx, int img_channels, const float* t, int64_t t_sb, int64_t t_sh,
                              int64_t t_sw, int B, int H, int W, int cout, const float* w, const float* bias,
                              const float* slope, int prec, void* out0, void* out1, int out_ctot, int32_t* sat_flag,
                              void* stream) {
  using namespace b200dn;
  B200DN_CHECK_ARG(x && w && bias && slope && out0, "conv_in: null pointer");
  B200DN_CHECK_ARG(B > 0 && Bx > 0 && H > 0 && W > 0, "conv_in: non-positive dims");
  B200DN_CHECK_ARG(img_channels == 3 || img_channels == 1, "conv_in: image channels must be 3 (RGB) or 1 (grayscale), got %d",
                   img_channels);
  B200DN_CHECK_ARG(cout > 0 && cout % 8 == 0, "conv_in: cout %d must be a multiple of 8", cout);
  B200DN_CHECK_ARG(out_ctot % 8 == 0 && out_ctot >= cout, "conv_in: out_ctot %d invalid", out_ctot);
  B200DN_CHECK_ARG(prec >= 0 && prec <= 4, "conv_in: bad prec %d", prec);
  const bool two = (prec == B200DN_PREC_BF16X2 || prec == B200DN_PREC_BF16X3 || prec == B200DN_PREC_FP16X2);
  B200DN_CHECK_ARG(!two || out1, "conv_in: prec %d needs the lo output plane", prec);
  B200DN_CHECK_ARG(B <= 65535 && H <= 65535 * 2 * ROWS * PASSES, "conv_in: B/H exceed the grid limit");
  if (int rc = require_sm100()) return rc;
  const int cin = img_channels + (t ? 1 : 0);
  const size_t smem = (static_cast<size_t>(cin) * 9 + 2) * cout * sizeof(float);
  B200DN_CHECK_ARG(smem <= 160 * 1024, "conv_in: cout %d too large", cout);
  dim3 block(PX, ROWS), grid(cdiv(W, PX), cdiv(H, 2 * ROWS * PASSES), B);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  uint16_t* o0 = static_cast<uint16_t*>(out0);
  uint16_t* o1 = two ? static_cast<uint16_t*>(out1) : nullptr;
  const bool single = prec == B200DN_PREC_BF16 || prec == B200DN_PREC_FP16;
  if (single && ingest_tc::enabled() && cout % 8 == 0 && cout <= ingest_tc::MAX_COUT) {
    // tensor-core ingest (single-plane modes): persistent grid, one CTA per SM
    // the sampler's call shape: two network images per input image, per-image scalar timesteps
    const bool twin = t != nullptr && B == 2 * Bx && t_sh == 0 && t_sw == 0 && H >= 2 && W >= 2 && ingest_tc::twin_enabled();
    const int tiles = (twin ? Bx : B) * cdiv(W, ingest_tc::TW_) * cdiv(H, ingest_tc::TH_);
    int sms = device_sm_count();
    if (sms <= 0) return B200DN_E_CUDA;
    const int g = tiles < sms ? tiles : sms;
    const bool bf = prec == B200DN_PREC_BF16;
    if (twin) {
      if (img_channels == 3)
        return ingest_tc::launch<3, true, true>(g, s, x, Bx, t, t_sb, t_sh, t_sw, B, H, W, cout, w, bias, slope, bf, o0, out_ctot, sat_flag);
      return ingest_tc::launch<1, true, true>(g, s, x, Bx, t, t_sb, t_sh, t_sw, B, H, W, cout, w, bias, slope, bf, o0, out_ctot, sat_flag);
    }
    if (img_channels == 3)
      return t ? ingest_tc::launch<3, true, false>(g, s, x, Bx, t, t_sb, t_sh, t_sw, B, H, W, cout, w, bias, slope, bf, o0, out_ctot, sat_flag)
               : ingest_tc::launch<3, false, false>(g, s, x, Bx, nullptr, 0, 0, 0, B, H, W, cout, w, bias, slope, bf, o0, out_ctot, sat_flag);
    return t ? ingest_tc::launch<1, true, false>(g, s, x, Bx, t, t_sb, t_sh, t_sw, B, H, W, cout, w, bias, slope, bf, o0, out_ctot, sat_flag)
             : ingest_tc::launch<1, false, false>(g, s, x, Bx, nullptr, 0, 0, 0, B, H, W, cout, w, bias, slope, bf, o0, out_ctot, sat_flag);
  }
  if (img_channels == 3)
    return t ? launch_conv_in<3, true>(grid, block, smem, s, x, Bx, t, t_sb, t_sh, t_sw, H, W, cout, w, bias, slope, prec, o0, o1, out_ctot, sat_flag)
             : launch_conv_in<3, false>(grid, block, smem, s, x, Bx, nullptr, 0, 0, 0, H, W, cout, w, bias, slope, prec, o0, o1, out_ctot, sat_flag);
  return t ? launch_conv_in<1, true>(grid, block, smem, s, x, Bx, t, t_sb, t_sh, t_sw, H, W, cout, w, bias, slope, prec, o0, o1, out_ctot, sat_flag)
           : launch_conv_in<1, false>(grid, block, smem, s, x, Bx, nullptr, 0, 0, 0, H, W, cout, w, bias, slope, prec, o0, o1, out_ctot, sat_flag);
}

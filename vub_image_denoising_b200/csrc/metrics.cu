// metrics.cu — on-device PSNR / SSIM reductions (128-bit loads, warp-shuffle block sums, fixed-order final sums).
//   PSNR: mse = mean((X-Y)^2); 10*log10(R^2/mse)          evaluate_Unet_diffusion/evaluate_model.py:36-41,
//                                                         evaluate_SIDD/evaluate_SIDD.py:63 (skimage PSNR)
//   SSIM: skimage.metrics.structural_similarity defaults   evaluate_Unet_diffusion/evaluate_model.py:30-34,
//         (scikit-image==0.22.0, requirements.txt:98)      evaluate_SIDD/evaluate_SIDD.py:64
// The kernels return raw sums (fp64); the host-side mirror turns them into dB / means, so a sharded run
// can all-reduce the sums.
//
// Reproducibility: every block writes ONE partial sum to a caller-provided workspace and a second kernel adds the
// partials of an image / plane in a fixed order, so the sums are bit-identical from run to run (the first version's
// atomicAdd(double) across blocks was not).
#include "common.cuh"

#include <array>
#include <utility>

namespace b200dn {

namespace {

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

template <int THREADS>
__device__ __forceinline__ double block_sum(double v, double* red) {
  v = warp_sum(v);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) red[warp] = v;
  __syncthreads();
  double t = 0.0;
  if (warp == 0) {
    t = (lane < THREADS / 32) ? red[lane] : 0.0;
    t = warp_sum(t);
  }
  return t;  // valid in warp 0
}

// out[i] = sum of partial[i * n_part + k], k = 0 .. n_part-1, in a fixed order (one warp per output).
__global__ void __launch_bounds__(128) sum_partials_kernel(const double* __restrict__ partial, int n_part, int64_t n_out,
                                                           double* __restrict__ out) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * 4 + (threadIdx.x >> 5);
  if (i >= n_out) return;
  const int lane = threadIdx.x & 31;
  const double* p = partial + i * n_part;
  double s = 0.0;
  for (int k = lane; k < n_part; k += 32) s += p[k];
  s = warp_sum(s);
  if (lane == 0) out[i] = s;
}

constexpr int SSE_THREADS = 256;
constexpr int SSE_MAX_CHUNKS = 1024;

// grid = (chunks, n_images); each block reduces a strided share of one image into one partial.
__global__ void __launch_bounds__(SSE_THREADS) sse_kernel(const float* __restrict__ a, const float* __restrict__ b,
                                                          int64_t n_per_image, int vec_ok, double* __restrict__ partial) {
  __shared__ double red[SSE_THREADS / 32];
  const int64_t img = blockIdx.y;
  const float* pa = a + img * n_per_image;
  const float* pb = b + img * n_per_image;
  float acc0 = 0.f, acc1 = 0.f, acc2 = 0.f, acc3 = 0.f;
  double dacc = 0.0;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * blockDim.x;
  const int64_t tid = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (vec_ok) {
    const int64_t n4 = n_per_image / 4;
    int it = 0;
    for (int64_t i = tid; i < n4; i += stride) {
      const float4 x = __ldg(reinterpret_cast<const float4*>(pa) + i);
      const float4 y = __ldg(reinterpret_cast<const float4*>(pb) + i);
      const float d0 = __fsub_rn(x.x, y.x), d1 = __fsub_rn(x.y, y.y), d2 = __fsub_rn(x.z, y.z), d3 = __fsub_rn(x.w, y.w);
      acc0 += __fmul_rn(d0, d0);
      acc1 += __fmul_rn(d1, d1);
      acc2 += __fmul_rn(d2, d2);
      acc3 += __fmul_rn(d3, d3);
      if (++it == 16) {  // spill the short fp32 partial sums into fp64 regularly
        dacc += static_cast<double>(acc0) + static_cast<double>(acc1) + static_cast<double>(acc2) + static_cast<double>(acc3);
        acc0 = acc1 = acc2 = acc3 = 0.f;
        it = 0;
      }
    }
    for (int64_t i = n4 * 4 + tid; i < n_per_image; i += stride) {
      const float d = __fsub_rn(pa[i], pb[i]);
      dacc += static_cast<double>(__fmul_rn(d, d));
    }
  } else {
    for (int64_t i = tid; i < n_per_image; i += stride) {
      const float d = __fsub_rn(pa[i], pb[i]);
      dacc += static_cast<double>(__fmul_rn(d, d));
    }
  }
  dacc += static_cast<double>(acc0) + static_cast<double>(acc1) + static_cast<double>(acc2) + static_cast<double>(acc3);
  const double t = block_sum<SSE_THREADS>(dacc, red);
  if (threadIdx.x == 0) partial[img * gridDim.x + blockIdx.x] = t;
}

int sse_chunks(int64_t n_images, int64_t n_per_image, int sms) {
  // enough blocks per image to cover the machine ~4x, at least 4 float4 per thread
  int64_t chunks = cdiv64(n_per_image / 4, static_cast<int64_t>(SSE_THREADS) * 4);
  const int64_t want = cdiv64(static_cast<int64_t>(sms) * 16, n_images);
  if (chunks > want) chunks = want;
  if (chunks > SSE_MAX_CHUNKS) chunks = SSE_MAX_CHUNKS;
  if (chunks < 1) chunks = 1;
  return static_cast<int>(chunks);
}

// ------------------------------------------------------------------ SSIM
// skimage 0.22 semantics: 7x7 uniform window (separable: axis 0 then axis 1), sample covariance (cov_norm = 49/48),
// K1 = 0.01, K2 = 0.03, crop 3, per-plane mean.
//
// One block (160 threads) = a 130 x 16 tile of the cropped output = a 136 x 22 input tile.
//   vertical pass:   thread = input column; its 22 x 2 samples come straight from global memory into registers
//                    (a warp reads 128 contiguous bytes per row; no input staging in shared memory), running 7-row sums
//                    of (x, y) and (x^2 + y^2, x*y) are written to shared memory as float2;
//   horizontal pass: half-warp = strip of 13 output columns, lane & 15 = row (odd pitch: conflict-free), running
//                    7-column sums, the SSIM map and its sum.
// Only FOUR window sums are needed, not skimage's five: vx and vy enter S only through vx + vy.  The sums run in fp32
// (add the entering / subtract the leaving sample, restarted every tile): skimage rounds each pass of scipy's
// double-accumulated uniform_filter to float32; fp32 sums differ from that by a few 1e-7 per mean with random sign,
// which moves the PLANE MEAN of S by < 1e-6 (tests hold 1e-5 against the oracle).  History: the first version kept
// fp64 sums and scalar loads into shared memory (0.09 of the HBM peak, F2F-conversion bound); an fp32 version that
// still staged inputs and five sums in shared memory reached 0.21, bound by ~0.9 shared-memory wavefronts per pixel;
// this layout needs ~0.36.
constexpr int TW = 130;                // output tile width: 130 + 120 cover the 250 output columns of a 256-wide patch
constexpr int TH = 16;                 // output tile height = rows of one half-warp in the horizontal pass
constexpr int NC = TW + 6;             // 136 input columns
constexpr int NR = TH + 6;             // 22 input rows
constexpr int PITCH = 137;             // odd: the lane-per-row walks of the horizontal pass are bank-conflict free
constexpr int SSIM_THREADS = 160;      // >= NC; 10 half-warps x 13 output columns
constexpr int STRIP = TW / (SSIM_THREADS / 16);   // 13
static_assert(STRIP * (SSIM_THREADS / 16) == TW && SSIM_THREADS >= NC, "ssim tile shape");

// Packed fp32 pairs (FADD2 / FFMA2: two IEEE fp32 operations per instruction on sm_100) carry the four window sums as
// (sum x, sum y) and (sum x^2 + y^2, sum x*y).
__device__ __forceinline__ float2 add2(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 sub2(float2 a, float2 b) { return __ffma2_rn(b, make_float2(-1.f, -1.f), a); }
__device__ __forceinline__ float2 moments(float2 xy) {   // (x^2 + y^2, x*y)
  return make_float2(fmaf(xy.x, xy.x, xy.y * xy.y), xy.x * xy.y);
}

// WC: compile-time image width (0 = runtime).  With WC = 256 — the patch size of every BASELINE configuration — the
// loads of the vertical pass are base + immediate offsets.  ncu on a 32-row-tile version (128 registers, 3 blocks =
// 15 warps per SM): issue slots 57 % busy, DRAM 33 %, shared memory 50 % — latency bound, a block alternates between
// waiting for its loads and computing; 16-row tiles halve the registers and the shared memory per block, so 5 blocks
// (25 warps) overlap those phases.
template <int WC>
__global__ void __launch_bounds__(SSIM_THREADS, 5) ssim_kernel(const float* __restrict__ a, const float* __restrict__ b,
                                                               int H, int W_rt, float C1, float C2, float cov_norm,
                                                               double* __restrict__ partial) {
  const int W = WC ? WC : W_rt;
  extern __shared__ float2 v[];         // [2][TH][PITCH]: vertical-pass 7-row SUMS of (x, y) and (x^2 + y^2, x*y)
  __shared__ double red[SSIM_THREADS / 32];
  constexpr int Q = TH * PITCH;

  const int64_t plane = blockIdx.z;
  const float* pa = a + plane * static_cast<int64_t>(H) * W;
  const float* pb = b + plane * static_cast<int64_t>(H) * W;
  const int oy0 = blockIdx.y * TH, ox0 = blockIdx.x * TW;  // origin in the cropped (H-6) x (W-6) output
  const int OH = H - 6, OW = W - 6;

  // ---- vertical pass: thread = input column, samples straight from global memory
  {
    const int c = threadIdx.x;
    const int gx = ox0 + c;
    if (c < NC) {
      float2 xy[NR];
      const float* qa = pa + static_cast<int64_t>(oy0) * W + gx;
      const float* qb = pb + static_cast<int64_t>(oy0) * W + gx;
      if (gx < W && oy0 + NR <= H) {       // interior tile: no per-sample bounds checks
#pragma unroll
        for (int k = 0; k < NR; ++k) xy[k] = make_float2(__ldg(qa + static_cast<int64_t>(k) * W), __ldg(qb + static_cast<int64_t>(k) * W));
      } else {
#pragma unroll
        for (int k = 0; k < NR; ++k) {
          const bool in = gx < W && oy0 + k < H;
          xy[k] = in ? make_float2(__ldg(qa + static_cast<int64_t>(k) * W), __ldg(qb + static_cast<int64_t>(k) * W))
                     : make_float2(0.f, 0.f);
        }
      }
      float2 s01 = make_float2(0.f, 0.f), s23 = s01;
#pragma unroll
      for (int k = 0; k < 6; ++k) {
        s01 = add2(s01, xy[k]);
        s23 = add2(s23, moments(xy[k]));
      }
#pragma unroll
      for (int o = 0; o < TH; ++o) {
        s01 = add2(s01, xy[o + 6]);
        s23 = add2(s23, moments(xy[o + 6]));
        v[o * PITCH + c] = s01;
        v[Q + o * PITCH + c] = s23;
        s01 = sub2(s01, xy[o]);
        s23 = sub2(s23, moments(xy[o]));
      }
    }
  }
  __syncthreads();

  // ---- horizontal pass + SSIM map: half-warp = strip of 13 output columns, lane & 15 = output row.
  // With S0..S3 the 49-sample sums: ux = S0/49, ..., and the constants folded into the FMAs:
  //   A1 = 2 ux uy + C1,  B1 = ux^2 + uy^2 + C1,  A2 = 2 cov (uxy - ux uy) + C2,  B2 = cov (uxx + uyy - ux^2 - uy^2) + C2
  float local = 0.f;
  {
    const int r = threadIdx.x & 15, c0 = (threadIdx.x >> 4) * STRIP;
    const int n_valid = OW - (ox0 + c0);
    if (oy0 + r < OH && n_valid > 0) {
      const float2* v0 = v + r * PITCH + c0;
      float2 w01[STRIP + 6], w23[STRIP + 6];
#pragma unroll
      for (int k = 0; k < STRIP + 6; ++k) {
        w01[k] = v0[k];
        w23[k] = v0[Q + k];
      }
      float2 s01 = make_float2(0.f, 0.f), s23 = s01;
#pragma unroll
      for (int k = 0; k < 6; ++k) s01 = add2(s01, w01[k]), s23 = add2(s23, w23[k]);
      constexpr float k1 = 1.0f / 49.0f, k2 = 1.0f / 2401.0f;
      const float ca = 2.f * cov_norm * k1, cb = -2.f * cov_norm * k2, cc = cov_norm * k1, cd = -cov_norm * k2;
#pragma unroll
      for (int o = 0; o < STRIP; ++o) {
        s01 = add2(s01, w01[o + 6]);
        s23 = add2(s23, w23[o + 6]);
        const float pxy = s01.x * s01.y;                       // 2401 ux uy
        const float m2 = fmaf(s01.x, s01.x, s01.y * s01.y);    // 2401 (ux^2 + uy^2)
        const float A1 = fmaf(pxy, 2.f * k2, C1);
        const float B1 = fmaf(m2, k2, C1);
        const float A2 = fmaf(s23.y, ca, fmaf(pxy, cb, C2));
        const float B2 = fmaf(s23.x, cc, fmaf(m2, cd, C2));
        float rden;   // B1 * B2 >= C1 * C2 > 0 and far from the denormal range: one MUFU.RCP, no range fix-up
        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rden) : "f"(B1 * B2));
        const float S = (A1 * A2) * rden;
        local += (o < n_valid) ? S : 0.f;
        s01 = sub2(s01, w01[o]);
        s23 = sub2(s23, w23[o]);
      }
    }
  }
  // a thread adds at most 13 values of |S| <= 1 in fp32; everything above that is summed in fp64
  const double t = block_sum<SSIM_THREADS>(static_cast<double>(local), red);
  if (threadIdx.x == 0)
    partial[(plane * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x] = t;
}

constexpr int SSIM_SMEM = 2 * TH * PITCH * static_cast<int>(sizeof(float2));
SmemOptIn g_ssim_opt_in;

// ------------------------------------------------------------------ SSIM, any separable window
// Every other option of skimage 0.22's structural_similarity: the 2R+1 taps of gaussian_filter (truncate 3.5) or
// uniform_filter (weights 1/win_size), scipy's 'reflect' borders, any cov_norm / C1 / C2, crop (win_size-1)/2 and an
// optional map of S.  ssim_kernel stays the only path of the default call; this kernel is its weighted generalisation.
// The taps differ, so there is no running sum: each output takes 2R+1 FFMA2 per pair of sums and pass.
//
// Same tile as ssim_kernel: one block (160 threads) = 130 x 16 outputs, an input tile of (130 + 2R) x (16 + 2R).
//   vertical pass:   thread = input column; it streams its 16 + 2R samples down from global memory and adds each
//                    into the sums of the output rows whose window holds it, so the registers do not grow with R
//                    (16 accumulator pairs); the weighted column sums of (x, y) and (x^2 + y^2, x*y) go to shared memory;
//   horizontal pass: half-warp = strip of 13 output columns, lane & 15 = row, streaming the 13 + 2R column sums.
// Outputs: the cropped region only (no map), or the whole plane (map).  Only tiles whose input window leaves the plane
// reflect their indices: the column once per thread, the rows through a per-block table.  Each output's sums are added in tap order from 0, so S at a pixel does not depend on the
// tiling, and a plane's partial sums do not depend on the batch.
struct SsimWindowParams {
  float w[2 * B200DN_SSIM_MAX_RADIUS + 1];
  float C1, C2, cov_norm;
  int pad;                 // crop (win_size - 1) / 2
};

// scipy.ndimage mode 'reflect' (d c b a | a b c d | d c b a): half-sample symmetric, periodic with period 2n, so any
// distance from the plane is folded back into it
__device__ __forceinline__ int reflect_index(int i, int n) {
  if (i >= 0 && i < n) return i;
  const int p = 2 * n;
  i %= p;
  if (i < 0) i += p;
  return i < n ? i : p - 1 - i;
}

__device__ __forceinline__ float2 fma2(float w, float2 x, float2 acc) { return __ffma2_rn(make_float2(w, w), x, acc); }

// vertical pass of one input column: sum over k of w[k] * sample(y0 + o + k), o = 0 .. TH-1, for (x, y) and the moments.
// EDGE: the tile's rows leave the plane; row k is rows[k], the reflected index.
template <int R, bool EDGE>
__device__ __forceinline__ void ssim_window_column(const float* __restrict__ pa, const float* __restrict__ pb, int gx,
                                                   int y0, const int* rows, int W, const SsimWindowParams& p,
                                                   float2* __restrict__ v01, float2* __restrict__ v23, int pitch) {
  float2 s01[TH], s23[TH];
#pragma unroll
  for (int o = 0; o < TH; ++o) s01[o] = s23[o] = make_float2(0.f, 0.f);
#pragma unroll
  for (int k = 0; k < TH + 2 * R; ++k) {
    const int64_t off = static_cast<int64_t>(EDGE ? rows[k] : y0 + k) * W + gx;
    const float2 xy = make_float2(__ldg(pa + off), __ldg(pb + off));
    const float2 m = moments(xy);
#pragma unroll
    for (int o = (k > 2 * R ? k - 2 * R : 0); o <= (k < TH - 1 ? k : TH - 1); ++o) {
      s01[o] = fma2(p.w[k - o], xy, s01[o]);
      s23[o] = fma2(p.w[k - o], m, s23[o]);
    }
  }
#pragma unroll
  for (int o = 0; o < TH; ++o) {
    v01[o * pitch] = s01[o];
    v23[o * pitch] = s23[o];
  }
}

// 4 blocks (20 warps) per SM: at ssim_kernel's 5 the 72-register cap spills the 16 accumulator pairs of the vertical pass
template <int R, bool MAP>
__global__ void __launch_bounds__(SSIM_THREADS, 4) ssim_window_kernel(const float* __restrict__ a,
                                                                      const float* __restrict__ b, int H, int W,
                                                                      const SsimWindowParams p, float* __restrict__ map,
                                                                      double* __restrict__ partial) {
  constexpr int NCW = TW + 2 * R;       // input columns of the tile
  constexpr int PW = NCW | 1;           // odd pitch: the lane-per-row walks of the horizontal pass are conflict free
  constexpr int Q = TH * PW;
  extern __shared__ float2 v[];         // [2][TH][PW]: weighted column sums of (x, y) and (x^2 + y^2, x*y)
  __shared__ double red[SSIM_THREADS / 32];
  __shared__ int rows[TH + 2 * R];

  const int64_t plane = blockIdx.z;
  const float* pa = a + plane * static_cast<int64_t>(H) * W;
  const float* pb = b + plane * static_cast<int64_t>(H) * W;
  const int base = MAP ? 0 : p.pad;     // outputs: the whole plane, or the cropped region
  const int oy0 = base + blockIdx.y * TH, ox0 = base + blockIdx.x * TW;   // plane coordinates of the first output
  const bool row_edge = oy0 < R || oy0 + TH + R > H;
  const bool col_edge = ox0 < R || ox0 + TW + R > W;
  if (row_edge) {   // a table, so that the loads of the vertical pass do not wait on the index arithmetic
    for (int k = threadIdx.x; k < TH + 2 * R; k += SSIM_THREADS) rows[k] = reflect_index(oy0 - R + k, H);
    __syncthreads();
  }

  {
    const int c = threadIdx.x;
    if (c < NCW) {
      const int gx = col_edge ? reflect_index(ox0 - R + c, W) : ox0 - R + c;
      if (row_edge)
        ssim_window_column<R, true>(pa, pb, gx, oy0 - R, rows, W, p, v + c, v + Q + c, PW);
      else
        ssim_window_column<R, false>(pa, pb, gx, oy0 - R, rows, W, p, v + c, v + Q + c, PW);
    }
  }
  __syncthreads();

  // horizontal pass + S (constants folded as in ssim_kernel; the weights sum to 1, so the sums are the means)
  const int r = threadIdx.x & 15, c0 = (threadIdx.x >> 4) * STRIP;
  const int gy = oy0 + r;
  const bool row_in = gy >= p.pad && gy < H - p.pad;
  float local = 0.f;
  float sv[STRIP];
  {
    const float2* v0 = v + r * PW + c0;
    float2 s01[STRIP], s23[STRIP];
#pragma unroll
    for (int o = 0; o < STRIP; ++o) s01[o] = s23[o] = make_float2(0.f, 0.f);
#pragma unroll
    for (int k = 0; k < STRIP + 2 * R; ++k) {
      const float2 w01 = v0[k], w23 = v0[Q + k];
#pragma unroll
      for (int o = (k > 2 * R ? k - 2 * R : 0); o <= (k < STRIP - 1 ? k : STRIP - 1); ++o) {
        s01[o] = fma2(p.w[k - o], w01, s01[o]);
        s23[o] = fma2(p.w[k - o], w23, s23[o]);
      }
    }
    const float ca = 2.f * p.cov_norm, cc = p.cov_norm;
#pragma unroll
    for (int o = 0; o < STRIP; ++o) {
      const float pxy = s01[o].x * s01[o].y;                        // ux uy
      const float m2 = fmaf(s01[o].x, s01[o].x, s01[o].y * s01[o].y);  // ux^2 + uy^2
      const float A1 = fmaf(pxy, 2.f, p.C1);
      const float B1 = m2 + p.C1;
      const float A2 = fmaf(s23[o].y, ca, fmaf(pxy, -ca, p.C2));
      const float B2 = fmaf(s23[o].x, cc, fmaf(m2, -cc, p.C2));
      const float S = (A1 * A2) / (B1 * B2);
      const int gx = ox0 + c0 + o;
      local += (row_in && gx >= p.pad && gx < W - p.pad) ? S : 0.f;
      sv[o] = S;
    }
  }
  if (MAP) {   // stage the tile's S in shared memory (v is consumed), then write whole rows
    constexpr int SP = TW + 1;
    static_assert(TH * SP <= 4 * Q, "the S tile fits in the sums' shared memory");
    float* st = reinterpret_cast<float*>(v);
    __syncthreads();
#pragma unroll
    for (int o = 0; o < STRIP; ++o) st[r * SP + c0 + o] = sv[o];
    __syncthreads();
    float* pm = map + plane * static_cast<int64_t>(H) * W;
    for (int i = threadIdx.x; i < TH * TW; i += SSIM_THREADS) {
      const int rr = i / TW, cc = i - rr * TW;
      const int y = oy0 + rr, x = ox0 + cc;
      if (y < H && x < W) pm[static_cast<int64_t>(y) * W + x] = st[rr * SP + cc];
    }
  }
  const double t = block_sum<SSIM_THREADS>(static_cast<double>(local), red);
  if (threadIdx.x == 0)
    partial[(plane * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x] = t;
}

template <int R>
int ssim_window_smem() { return 2 * TH * ((TW + 2 * R) | 1) * static_cast<int>(sizeof(float2)); }

using SsimWindowLaunch = void (*)(dim3, cudaStream_t, const float*, const float*, int, int, const SsimWindowParams&,
                                  float*, double*);
template <int R>
void launch_ssim_window(dim3 grid, cudaStream_t s, const float* a, const float* b, int H, int W,
                        const SsimWindowParams& p, float* map, double* partial) {
  static_assert(2 * TH * ((TW + 2 * R) | 1) * sizeof(float2) <= 48 * 1024, "no shared-memory opt-in needed");
  if (map)
    ssim_window_kernel<R, true><<<grid, SSIM_THREADS, ssim_window_smem<R>(), s>>>(a, b, H, W, p, map, partial);
  else
    ssim_window_kernel<R, false><<<grid, SSIM_THREADS, ssim_window_smem<R>(), s>>>(a, b, H, W, p, map, partial);
}
template <int... Rs>
constexpr std::array<SsimWindowLaunch, sizeof...(Rs)> ssim_window_launchers(std::integer_sequence<int, Rs...>) {
  return {&launch_ssim_window<Rs>...};
}
static_assert(TW + 2 * B200DN_SSIM_MAX_RADIUS <= SSIM_THREADS, "one thread per input column");

}  // namespace
}  // namespace b200dn

extern "C" int64_t b200dn_psnr_sse_workspace_bytes(int64_t n_images, int64_t n_per_image) {
  if (n_images <= 0 || n_per_image <= 0) return 0;
  return n_images * b200dn::SSE_MAX_CHUNKS * static_cast<int64_t>(sizeof(double));
}

extern "C" int64_t b200dn_ssim_workspace_bytes(int64_t n_planes, int H, int W) {
  using namespace b200dn;
  if (n_planes <= 0 || H < 7 || W < 7) return 0;
  return n_planes * cdiv(W - 6, TW) * cdiv(H - 6, TH) * static_cast<int64_t>(sizeof(double));
}

extern "C" int b200dn_psnr_sse(const float* a, const float* b, int64_t n_images, int64_t n_per_image, double* sse,
                               void* workspace, int64_t workspace_bytes, void* stream) {
  using namespace b200dn;
  B200DN_CHECK_ARG(a && b && sse && n_images > 0 && n_per_image > 0, "psnr_sse: bad arguments");
  B200DN_CHECK_ARG(n_images <= 65535, "psnr_sse: at most 65535 images per call");
  if (int rc = require_sm100()) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int vec_ok = ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b)) & 15) == 0 && (n_per_image % 4 == 0);
  int sms = device_sm_count();
  if (sms <= 0) return B200DN_E_CUDA;
  const int chunks = sse_chunks(n_images, n_per_image, sms);
  B200DN_CHECK_ARG(workspace && (reinterpret_cast<uintptr_t>(workspace) & 7) == 0 &&
                       workspace_bytes >= n_images * chunks * static_cast<int64_t>(sizeof(double)),
                   "psnr_sse: workspace of b200dn_psnr_sse_workspace_bytes() bytes (8-byte aligned) required");
  double* partial = static_cast<double*>(workspace);
  dim3 grid(static_cast<unsigned>(chunks), static_cast<unsigned>(n_images));
  sse_kernel<<<grid, SSE_THREADS, 0, s>>>(a, b, n_per_image, vec_ok, partial);
  B200DN_CUDA(cudaGetLastError());
  sum_partials_kernel<<<static_cast<unsigned>(cdiv64(n_images, 4)), 128, 0, s>>>(partial, chunks, n_images, sse);
  B200DN_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int b200dn_ssim(const float* a, const float* b, int64_t n_planes, int H, int W, float data_range,
                           double* ssim_sum, void* workspace, int64_t workspace_bytes, void* stream) {
  using namespace b200dn;
  B200DN_CHECK_ARG(a && b && ssim_sum && n_planes > 0, "ssim: bad arguments");
  B200DN_CHECK_ARG(H >= 7 && W >= 7, "ssim: win_size 7 exceeds image extent %d x %d", H, W);
  B200DN_CHECK_ARG(n_planes <= 65535, "ssim: at most 65535 planes per call");
  B200DN_CHECK_ARG(workspace && (reinterpret_cast<uintptr_t>(workspace) & 7) == 0 &&
                       workspace_bytes >= b200dn_ssim_workspace_bytes(n_planes, H, W),
                   "ssim: workspace of b200dn_ssim_workspace_bytes() bytes (8-byte aligned) required");
  if (int rc = require_sm100()) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  static const void* const kernels[2] = {reinterpret_cast<const void*>(ssim_kernel<0>),
                                         reinterpret_cast<const void*>(ssim_kernel<256>)};
  if (int rc = ensure_max_dyn_smem(g_ssim_opt_in, kernels, 2, SSIM_SMEM, "cudaFuncSetAttribute(ssim_kernel, smem)")) return rc;
  // python: C1 = (K1*R)**2 in double, then used against float32 arrays (NEP 50 weak scalar -> float32)
  const double R = static_cast<double>(data_range);
  const float C1 = static_cast<float>((0.01 * R) * (0.01 * R));
  const float C2 = static_cast<float>((0.03 * R) * (0.03 * R));
  const float cov_norm = static_cast<float>(49.0 / 48.0);
  dim3 grid(cdiv(W - 6, TW), cdiv(H - 6, TH), static_cast<unsigned>(n_planes));
  double* partial = static_cast<double*>(workspace);
  if (W == 256)
    ssim_kernel<256><<<grid, SSIM_THREADS, SSIM_SMEM, s>>>(a, b, H, W, C1, C2, cov_norm, partial);
  else
    ssim_kernel<0><<<grid, SSIM_THREADS, SSIM_SMEM, s>>>(a, b, H, W, C1, C2, cov_norm, partial);
  B200DN_CUDA(cudaGetLastError());
  sum_partials_kernel<<<static_cast<unsigned>(cdiv64(n_planes, 4)), 128, 0, s>>>(partial, grid.x * grid.y, n_planes, ssim_sum);
  B200DN_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int64_t b200dn_ssim_window_workspace_bytes(int64_t n_planes, int H, int W) {
  using namespace b200dn;
  if (n_planes <= 0 || H < 1 || W < 1) return 0;
  // the tiling of the whole plane (map) has at least as many tiles as that of the cropped region
  return n_planes * cdiv(W, TW) * cdiv(H, TH) * static_cast<int64_t>(sizeof(double));
}

extern "C" int b200dn_ssim_window(const float* a, const float* b, int64_t n_planes, int H, int W,
                                  const b200dn_ssim_window_opts* opts, double* ssim_sum, float* map, void* workspace,
                                  int64_t workspace_bytes, void* stream) {
  using namespace b200dn;
  B200DN_CHECK_ARG(a && b && opts && ssim_sum && n_planes > 0 && H > 0 && W > 0, "ssim_window: bad arguments");
  B200DN_CHECK_ARG(opts->radius >= 0 && opts->radius <= B200DN_SSIM_MAX_RADIUS,
                   "ssim_window: filter radius %d outside 0..%d", opts->radius, B200DN_SSIM_MAX_RADIUS);
  B200DN_CHECK_ARG(opts->win_size >= 1 && opts->win_size % 2 == 1, "ssim_window: win_size %d must be odd",
                   opts->win_size);
  B200DN_CHECK_ARG(opts->win_size <= H && opts->win_size <= W, "ssim_window: win_size %d exceeds image extent %d x %d",
                   opts->win_size, H, W);
  B200DN_CHECK_ARG(n_planes <= 65535, "ssim_window: at most 65535 planes per call");
  B200DN_CHECK_ARG(workspace && (reinterpret_cast<uintptr_t>(workspace) & 7) == 0 &&
                       workspace_bytes >= b200dn_ssim_window_workspace_bytes(n_planes, H, W),
                   "ssim_window: workspace of b200dn_ssim_window_workspace_bytes() bytes (8-byte aligned) required");
  if (int rc = require_sm100()) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  SsimWindowParams p;
  for (int k = 0; k < 2 * B200DN_SSIM_MAX_RADIUS + 1; ++k) p.w[k] = k <= 2 * opts->radius ? opts->weights[k] : 0.f;
  p.C1 = opts->C1;
  p.C2 = opts->C2;
  p.cov_norm = opts->cov_norm;
  p.pad = (opts->win_size - 1) / 2;
  const int OH = map ? H : H - 2 * p.pad, OW = map ? W : W - 2 * p.pad;
  dim3 grid(cdiv(OW, TW), cdiv(OH, TH), static_cast<unsigned>(n_planes));
  static constexpr auto launchers = ssim_window_launchers(std::make_integer_sequence<int, B200DN_SSIM_MAX_RADIUS + 1>{});
  double* partial = static_cast<double*>(workspace);
  launchers[opts->radius](grid, s, a, b, H, W, p, map, partial);
  B200DN_CUDA(cudaGetLastError());
  sum_partials_kernel<<<static_cast<unsigned>(cdiv64(n_planes, 4)), 128, 0, s>>>(partial, grid.x * grid.y, n_planes, ssim_sum);
  B200DN_CUDA(cudaGetLastError());
  return 0;
}

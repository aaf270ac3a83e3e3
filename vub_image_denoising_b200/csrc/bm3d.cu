// bm3d.cu — BM3D / CBM3D denoising (b200dn.h, "BM3D / CBM3D").  One stage is four launches on the caller's stream:
//   bm3d_ingest_kernel : RGB (or grey) fp32 -> fp64 opponent planes, and the int32 matching plane q = rint(1024 Y)
//                        with Y = ((R + G) + B) * fl32(1/3) in fp32 (grey: Y = z)
//   bm3d_match_kernel  : one warp per reference block, eight reference blocks of one row per block; the search region
//                        of the eight sits in shared memory, each lane keeps its own sorted top-(N2 - 1) list of packed
//                        (d, window position) keys, and a warp merge picks the group
//   bm3d_filter_kernel : one block per group and stage: gather, 2-D DCT, Haar along the group, hard threshold (stage 1)
//                        or Wiener shrinkage against the basic estimate (stage 2), inverse, Kaiser-weighted sums
//   bm3d_finish_kernel : numerator / denominator, inverse opponent transform, fp32 NCHW out
// The filter runs in fp64: a hard-threshold decision flips on an absolute coefficient error of 2.7 sigma_c * 1e-5
// (3e-7 at sigma = 10/255), and an fp32 group transform of a 32-block group is off by about 1e-6 there.  The sums are
// 64-bit fixed point at 2^-32 (integer atomics commute, so the output does not depend on the order of the groups).
#include "common.cuh"

namespace b200dn {

namespace {

constexpr int BS = 8;                  // block edge
constexpr int NS_HALF = 19;            // search radius (Ns = 39)
constexpr int NS = 2 * NS_HALF + 1;
constexpr int MATCH_WARPS = 8;         // reference blocks (one row) per match block
constexpr int REGION_ROWS = 2 * NS_HALF + BS;                                    // 46
constexpr int REGION_COLS = 3 * (MATCH_WARPS - 1) + 2 * NS_HALF + BS;            // 67
constexpr int FILTER_THREADS = 128;
constexpr unsigned DIFF_CLAMP = 4096;  // |q_R - q| above this rejects anyway (4096^2 > tau); keeps d < 2^31
constexpr double FIX_SCALE = 4294967296.0;   // 2^32
constexpr double LAMBDA_HARD = 2.7;
constexpr double WIENER_FLOOR = 1.0 / 1024.0;
constexpr int TAU_HT = 3096141;        // floor(3000 * 64 * 2^20 / 255^2)
constexpr int TAU_WIE = 412818;        // floor(400 * 64 * 2^20 / 255^2)

// np.kaiser(8, 2.0)
__constant__ double c_kaiser[BS] = {0x1.c1345acdb96a2p-2, 0x1.5cd688a740b7cp-1, 0x1.c0f128fa38683p-1,
                                    0x1.f8bdba3f962acp-1, 0x1.f8bdba3f962acp-1, 0x1.c0f128fa38683p-1,
                                    0x1.5cd688a740b7cp-1, 0x1.c1345acdb96a2p-2};

__host__ __device__ __forceinline__ int nref(int n) { return B200DN_BM3D_NREF(n); }
__device__ __forceinline__ int ref_pos(int i, int n) { return i < (n - BS) / 3 + 1 ? 3 * i : n - BS; }

// ||A_c||_2 of the opponent rows (1/3, 1/3, 1/3), (1/2, 0, -1/2), (1/4, -1/2, 1/4); 1 for grey
__device__ __forceinline__ double channel_norm(int C, int c) {
  if (C == 1) return 1.0;
  return c == 0 ? sqrt(1.0 / 3.0) : (c == 1 ? sqrt(0.5) : sqrt(0.375));
}

// src [B, C, H, W] fp32 -> planes [B, C, H, W] fp64 (opponent for C = 3), q [B, H, W] (optional)
__global__ void bm3d_ingest_kernel(const float* __restrict__ src, int64_t pixels, int C, int64_t hw,
                                   double* __restrict__ planes, int* __restrict__ q) {
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < pixels;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t b = i / hw, p = i - b * hw;
    const float* s = src + b * C * hw + p;
    double* o = planes + b * C * hw + p;
    float y;
    if (C == 1) {
      y = s[0];
      o[0] = y;
    } else {
      const float r = s[0], g = s[hw], bl = s[2 * hw];
      y = __fmul_rn(__fadd_rn(__fadd_rn(r, g), bl), 1.0f / 3.0f);
      const double R = r, G = g, Bd = bl;
      o[0] = (R + G + Bd) / 3.0;
      o[hw] = (R - Bd) * 0.5;
      o[2 * hw] = (R + Bd) * 0.25 - G * 0.5;
    }
    if (q) q[i] = __float2int_rn(__fmul_rn(y, 1024.0f));
  }
}

// Grid (cdiv(nC, 8), nR, B); warp w matches reference block (blockIdx.y, blockIdx.x * 8 + w).
template <int N2>
__global__ void __launch_bounds__(32 * MATCH_WARPS) bm3d_match_kernel(const int* __restrict__ q, int H, int W, int tau,
                                                                     int* __restrict__ match, int* __restrict__ gsize) {
  constexpr int K = N2 - 1;
  constexpr unsigned long long NONE = ~0ull;
  __shared__ int S[REGION_ROWS][REGION_COLS + 1];
  const int nR = nref(H), nC = nref(W);
  const int b = blockIdx.z, ir = blockIdx.y, warp = threadIdx.x / 32, lane = threadIdx.x % 32;
  const int jc0 = blockIdx.x * MATCH_WARPS;
  const int jc_last = min(jc0 + MATCH_WARPS, nC) - 1;
  const int rr = ref_pos(ir, H);
  const int r_lo = max(0, rr - NS_HALF), r_hi = min(H - BS, rr + NS_HALF) + BS;                       // [r_lo, r_hi)
  const int c_lo = max(0, ref_pos(jc0, W) - NS_HALF), c_hi = min(W - BS, ref_pos(jc_last, W) + NS_HALF) + BS;
  const int rows = r_hi - r_lo, cols = c_hi - c_lo;
  const int* qb = q + static_cast<int64_t>(b) * H * W;
  for (int e = threadIdx.x; e < rows * cols; e += blockDim.x) {
    const int i = e / cols, j = e - i * cols;
    S[i][j] = __ldg(qb + static_cast<int64_t>(r_lo + i) * W + c_lo + j);
  }
  __syncthreads();
  const int jc = jc0 + warp;
  if (jc >= nC) return;
  const int rc = ref_pos(jc, W);
  const int cr_lo = max(0, rr - NS_HALF), cr_hi = min(H - BS, rr + NS_HALF);      // candidate corners, inclusive
  const int cc_lo = max(0, rc - NS_HALF), cc_hi = min(W - BS, rc + NS_HALF);
  const int ncc = cc_hi - cc_lo + 1, ncand = (cr_hi - cr_lo + 1) * ncc;
  const int ri = rr - r_lo, ci = rc - c_lo;
  unsigned long long L[K];
#pragma unroll
  for (int k = 0; k < K; ++k) L[k] = NONE;
  for (int e = lane; e < ncand; e += 32) {
    const int dr = e / ncc, dc = e - dr * ncc;
    const int r = cr_lo + dr, c = cc_lo + dc;
    if (r == rr && c == rc) continue;
    const int si = r - r_lo, sj = c - c_lo;
    unsigned d = 0;
#pragma unroll
    for (int i = 0; i < BS; ++i)
#pragma unroll
      for (int j = 0; j < BS; ++j) {
        const unsigned a = min(__sad(S[si + i][sj + j], S[ri + i][ci + j], 0u), DIFF_CLAMP);
        d += a * a;
      }
    if (d > static_cast<unsigned>(tau)) continue;
    // (d, r, c) order == (d, window position) order: the window position is row-major in (r - rr, c - rc)
    const unsigned long long key = (static_cast<unsigned long long>(d) << 11) |
                                   static_cast<unsigned>((r - rr + NS_HALF) * NS + (c - rc + NS_HALF));
    if (key < L[K - 1]) {
#pragma unroll
      for (int k = K - 1; k > 0; --k) L[k] = L[k] < key ? L[k] : (L[k - 1] > key ? L[k - 1] : key);
      L[0] = L[0] < key ? L[0] : key;
    }
  }
  // warp merge: K rounds of the smallest list head (keys are distinct, so exactly one lane pops)
  const int64_t g = (static_cast<int64_t>(b) * nR + ir) * nC + jc;
  int* out = match + g * N2;
  int n = 1;
  if (lane == 0) out[0] = rr * W + rc;
  for (int k = 0; k < K; ++k) {
    unsigned long long m = L[0];
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      const unsigned long long o = __shfl_xor_sync(0xffffffffu, m, off);
      m = o < m ? o : m;
    }
    if (m == NONE) break;
    if (L[0] == m) {
#pragma unroll
      for (int i = 0; i < K - 1; ++i) L[i] = L[i + 1];
      L[K - 1] = NONE;
    }
    const int wpos = static_cast<int>(m & 2047u);
    if (lane == 0) out[n] = (rr + wpos / NS - NS_HALF) * W + rc + wpos % NS - NS_HALF;
    ++n;
  }
  int n2 = 1;
  while (2 * n2 <= n) n2 *= 2;
  for (int k = n2 + lane; k < N2; k += 32) out[k] = -1;
  if (lane == 0) gsize[g] = n2;
}

// Orthonormal Haar along the group (length n, a power of two <= N) on a register vector: H_2m = (1/sqrt 2) [H_m (x) [1, 1];
// I_m (x) [1, -1]], i.e. the first half of every level is the pairwise sums, the second half the differences.
template <int N>
__device__ __forceinline__ void haar_fwd(double (&v)[N], int n) {
#pragma unroll
  for (int len = N; len > 1; len >>= 1) {
    if (len <= n) {
      double t[N];
#pragma unroll
      for (int i = 0; i < len / 2; ++i) {
        t[i] = (v[2 * i] + v[2 * i + 1]) * M_SQRT1_2;
        t[len / 2 + i] = (v[2 * i] - v[2 * i + 1]) * M_SQRT1_2;
      }
#pragma unroll
      for (int i = 0; i < len; ++i) v[i] = t[i];
    }
  }
}
template <int N>
__device__ __forceinline__ void haar_inv(double (&v)[N], int n) {
#pragma unroll
  for (int len = 2; len <= N; len <<= 1) {
    if (len <= n) {
      double t[N];
#pragma unroll
      for (int i = 0; i < len / 2; ++i) {
        t[2 * i] = (v[i] + v[len / 2 + i]) * M_SQRT1_2;
        t[2 * i + 1] = (v[i] - v[len / 2 + i]) * M_SQRT1_2;
      }
#pragma unroll
      for (int i = 0; i < len; ++i) v[i] = t[i];
    }
  }
}

// In-place separable 8 x 8 transform of n blocks X[g][64]: rows then columns, with D (inverse: D^T).
template <bool INV>
__device__ __forceinline__ void dct2(double* X, int n, const double (&D)[BS][BS]) {
  for (int e = threadIdx.x; e < n * BS; e += blockDim.x) {              // row e % 8 of block e / 8
    double* p = X + (e / BS) * 64 + (e % BS) * BS;
    double in[BS], o[BS];
#pragma unroll
    for (int j = 0; j < BS; ++j) in[j] = p[j];
#pragma unroll
    for (int k = 0; k < BS; ++k) {
      double a = 0.0;
#pragma unroll
      for (int j = 0; j < BS; ++j) a = fma(INV ? D[j][k] : D[k][j], in[j], a);
      o[k] = a;
    }
#pragma unroll
    for (int k = 0; k < BS; ++k) p[k] = o[k];
  }
  __syncthreads();
  for (int e = threadIdx.x; e < n * BS; e += blockDim.x) {              // column e % 8 of block e / 8
    double* p = X + (e / BS) * 64 + (e % BS);
    double in[BS], o[BS];
#pragma unroll
    for (int i = 0; i < BS; ++i) in[i] = p[i * BS];
#pragma unroll
    for (int k = 0; k < BS; ++k) {
      double a = 0.0;
#pragma unroll
      for (int i = 0; i < BS; ++i) a = fma(INV ? D[i][k] : D[k][i], in[i], a);
      o[k] = a;
    }
#pragma unroll
    for (int k = 0; k < BS; ++k) p[k * BS] = o[k];
  }
  __syncthreads();
}

// Deterministic block sum of one value per thread (fixed shuffle tree, then the warps in order).
__device__ __forceinline__ double block_sum(double v, double* red) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
  if (threadIdx.x % 32 == 0) red[threadIdx.x / 32] = v;
  __syncthreads();
  double s = 0.0;
  for (int w = 0; w < FILTER_THREADS / 32; ++w) s += red[w];
  __syncthreads();
  return s;
}

// Grid (nC, nR, B): one group.  STAGE 1: hard thresholding of the noisy planes; STAGE 2: Wiener shrinkage of the
// noisy planes against the basic planes.  num / den [B, C, H, W] collect w K x and w K in 2^-32 fixed point.
template <int STAGE, int N2>
__global__ void __launch_bounds__(FILTER_THREADS) bm3d_filter_kernel(
    const double* __restrict__ planes, const double* __restrict__ bplanes, const int* __restrict__ match,
    const int* __restrict__ gsize, const float* __restrict__ sigma, int C, int H, int W,
    unsigned long long* __restrict__ num, unsigned long long* __restrict__ den) {
  __shared__ double X[N2 * 64];
  __shared__ double Wb[STAGE == 2 ? N2 * 64 : 1];
  __shared__ double D[BS][BS];
  __shared__ double Kw[64];                    // Kaiser window k k^T
  __shared__ double red[FILTER_THREADS / 32];
  __shared__ int pos[N2];
  const int nR = gridDim.y, nC = gridDim.x, b = blockIdx.z;
  const int64_t g = (static_cast<int64_t>(b) * nR + blockIdx.y) * nC + blockIdx.x;
  const int n = gsize[g];
  const int t = threadIdx.x;
  if (t < 64) {
    const int k = t / BS, j = t % BS;
    D[k][j] = (k == 0 ? sqrt(0.125) : 0.5) * cospi((2 * j + 1) * k / 16.0);
    Kw[t] = c_kaiser[k] * c_kaiser[j];
  }
  if (t < N2) pos[t] = match[g * N2 + t];
  __syncthreads();
  const int64_t hw = static_cast<int64_t>(H) * W;
  const double sig = sigma[b];
  for (int c = 0; c < C; ++c) {
    const int64_t plane = (static_cast<int64_t>(b) * C + c) * hw;
    const double sc = sig * channel_norm(C, c);
    for (int e = t; e < n * 64; e += FILTER_THREADS) {
      const int p = pos[e / 64], i = (e % 64) / BS, j = e % BS;
      const int64_t at = plane + p + static_cast<int64_t>(i) * W + j;
      X[e] = planes[at];
      if constexpr (STAGE == 2) Wb[e] = bplanes[at];
    }
    __syncthreads();
    dct2<false>(X, n, D);
    if constexpr (STAGE == 2) dct2<false>(Wb, n, D);
    // along the group: thread t < 64 owns coefficient t of every block
    double part = 0.0;
    if (t < 64) {
      double v[N2];
      if constexpr (STAGE == 2) {
        // Wb <- W = gb^2 / (gb^2 + sigma_c^2)
#pragma unroll
        for (int k = 0; k < N2; ++k) v[k] = k < n ? Wb[k * 64 + t] : 0.0;
        haar_fwd<N2>(v, n);
        const double s2 = sc * sc;
#pragma unroll
        for (int k = 0; k < N2; ++k)
          if (k < n) {
            const double w = v[k] * v[k] / (v[k] * v[k] + s2);
            Wb[k * 64 + t] = w;
            part += w * w;
          }
      }
#pragma unroll
      for (int k = 0; k < N2; ++k) v[k] = k < n ? X[k * 64 + t] : 0.0;
      haar_fwd<N2>(v, n);
      if constexpr (STAGE == 1) {
        const double thr = LAMBDA_HARD * sc;
#pragma unroll
        for (int k = 0; k < N2; ++k) {
          const bool keep = fabs(v[k]) > thr;
          v[k] = keep ? v[k] : 0.0;
          part += (k < n && keep) ? 1.0 : 0.0;
        }
      } else {
#pragma unroll
        for (int k = 0; k < N2; ++k) v[k] = k < n ? v[k] * Wb[k * 64 + t] : 0.0;
      }
      haar_inv<N2>(v, n);
#pragma unroll
      for (int k = 0; k < N2; ++k)
        if (k < n) X[k * 64 + t] = v[k];
    }
    const double s = block_sum(part, red);       // N_har (exact) or ||W||^2; includes a __syncthreads
    const double wgt = STAGE == 1 ? 1.0 / fmax(s, 1.0) : 1.0 / fmax(s, WIENER_FLOOR);
    dct2<true>(X, n, D);
    for (int e = t; e < n * 64; e += FILTER_THREADS) {
      const int p = pos[e / 64], i = (e % 64) / BS, j = e % BS;
      const int64_t at = plane + p + static_cast<int64_t>(i) * W + j;
      const double wk = wgt * Kw[e % 64];
      atomicAdd(num + at, static_cast<unsigned long long>(__double2ll_rn(wk * X[e] * FIX_SCALE)));
      atomicAdd(den + at, static_cast<unsigned long long>(__double2ll_rn(wk * FIX_SCALE)));
    }
    __syncthreads();
  }
}

// out [B, C, H, W] fp32 = inverse opponent of num / den
__global__ void bm3d_finish_kernel(const long long* __restrict__ num, const long long* __restrict__ den,
                                   int64_t pixels, int C, int64_t hw, float* __restrict__ out) {
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < pixels;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t b = i / hw, p = i - b * hw, at = b * C * hw + p;
    if (C == 1) {
      out[at] = static_cast<float>(static_cast<double>(num[at]) / static_cast<double>(den[at]));
    } else {
      const double y = static_cast<double>(num[at]) / static_cast<double>(den[at]);
      const double u = static_cast<double>(num[at + hw]) / static_cast<double>(den[at + hw]);
      const double v = static_cast<double>(num[at + 2 * hw]) / static_cast<double>(den[at + 2 * hw]);
      out[at] = static_cast<float>(y + u + v * (2.0 / 3.0));
      out[at + hw] = static_cast<float>(y - v * (4.0 / 3.0));
      out[at + 2 * hw] = static_cast<float>(y - u + v * (2.0 / 3.0));
    }
  }
}

struct Workspace {
  double *planes, *bplanes;
  long long *num, *den;
  float* basic;
  int *q, *match, *gsize;
  int64_t bytes;
};

Workspace carve(const b200dn_bm3d_args& a, char* base) {
  const int64_t px = static_cast<int64_t>(a.B) * a.H * a.W, vals = px * a.C;
  const int64_t groups = static_cast<int64_t>(a.B) * nref(a.H) * nref(a.W);
  Workspace w{};
  int64_t off = 0;
  auto take = [&](int64_t bytes) {
    char* p = base ? base + off : nullptr;
    off += (bytes + 255) / 256 * 256;
    return p;
  };
  w.planes = reinterpret_cast<double*>(take(vals * 8));
  w.bplanes = reinterpret_cast<double*>(take(vals * 8));
  w.num = reinterpret_cast<long long*>(take(vals * 8));
  w.den = reinterpret_cast<long long*>(take(vals * 8));
  w.basic = reinterpret_cast<float*>(take(vals * 4));
  w.q = reinterpret_cast<int*>(take(px * 4));
  w.match = reinterpret_cast<int*>(take(groups * B200DN_BM3D_N2_WIE * 4));
  w.gsize = reinterpret_cast<int*>(take(groups * 4));
  w.bytes = off;
  return w;
}

int grid_1d(int64_t n) { return static_cast<int>(n / 256 + 1 < 65536 * 8 ? n / 256 + 1 : 65536 * 8); }

// one stage: STAGE 1 filters z's planes on groups matched on z; STAGE 2 filters them against `basic`'s planes on groups
// matched on basic.  Writes out (fp32 RGB / grey) and, when given, the groups.
template <int STAGE>
int run_stage(const b200dn_bm3d_args& a, const Workspace& w, const float* basic, float* out, int* match, int* gsize,
              cudaStream_t s) {
  constexpr int N2 = STAGE == 1 ? B200DN_BM3D_N2_HT : B200DN_BM3D_N2_WIE;
  const int64_t hw = static_cast<int64_t>(a.H) * a.W, px = a.B * hw, vals = px * a.C;
  bm3d_ingest_kernel<<<grid_1d(px), 256, 0, s>>>(a.z, px, a.C, hw, w.planes, STAGE == 1 ? w.q : nullptr);
  if (STAGE == 2) bm3d_ingest_kernel<<<grid_1d(px), 256, 0, s>>>(basic, px, a.C, hw, w.bplanes, w.q);
  B200DN_CUDA(cudaMemsetAsync(w.num, 0, vals * 8, s));
  B200DN_CUDA(cudaMemsetAsync(w.den, 0, vals * 8, s));
  const int nR = nref(a.H), nC = nref(a.W);
  bm3d_match_kernel<N2><<<dim3(cdiv(nC, MATCH_WARPS), nR, a.B), 32 * MATCH_WARPS, 0, s>>>(
      w.q, a.H, a.W, STAGE == 1 ? TAU_HT : TAU_WIE, match ? match : w.match, gsize ? gsize : w.gsize);
  bm3d_filter_kernel<STAGE, N2><<<dim3(nC, nR, a.B), FILTER_THREADS, 0, s>>>(
      w.planes, w.bplanes, match ? match : w.match, gsize ? gsize : w.gsize, a.sigma, a.C, a.H, a.W,
      reinterpret_cast<unsigned long long*>(w.num), reinterpret_cast<unsigned long long*>(w.den));
  bm3d_finish_kernel<<<grid_1d(px), 256, 0, s>>>(w.num, w.den, px, a.C, hw, out);
  B200DN_CUDA(cudaGetLastError());
  return 0;
}

int check_args(const b200dn_bm3d_args* a) {
  B200DN_CHECK_ARG(a, "bm3d: null args");
  B200DN_CHECK_ARG(a->z && a->sigma && a->out, "bm3d: z, sigma and out are required");
  B200DN_CHECK_ARG(a->B > 0 && (a->C == 1 || a->C == 3) && a->H >= BS && a->W >= BS,
                   "bm3d: bad shape [%d, %d, %d, %d] (C must be 1 or 3, H and W at least 8)", a->B, a->C, a->H, a->W);
  B200DN_CHECK_ARG(static_cast<int64_t>(a->H) * a->W < (int64_t{1} << 31) && a->B <= 65535 && nref(a->H) <= 65535,
                   "bm3d: image too large [%d, %d, %d]", a->B, a->H, a->W);
  B200DN_CHECK_ARG(a->stages == B200DN_BM3D_HARD_THRESHOLDING || a->stages == B200DN_BM3D_ALL_STAGES,
                   "bm3d: stages must be 1 (hard thresholding) or 3 (all stages), got %d", a->stages);
  B200DN_CHECK_ARG(!a->basic || a->stages == B200DN_BM3D_ALL_STAGES,
                   "bm3d: a basic estimate runs stage 2, which stages = 1 excludes");
  return 0;
}

}  // namespace
}  // namespace b200dn

extern "C" int64_t b200dn_bm3d_workspace_bytes(const b200dn_bm3d_args* args) {
  using namespace b200dn;
  if (int rc = check_args(args)) return rc;
  return carve(*args, nullptr).bytes;
}

extern "C" int b200dn_bm3d(const b200dn_bm3d_args* args, void* workspace, int64_t workspace_bytes, void* stream) {
  using namespace b200dn;
  if (int rc = check_args(args)) return rc;
  const b200dn_bm3d_args& a = *args;
  const Workspace w = carve(a, static_cast<char*>(workspace));
  B200DN_CHECK_ARG(workspace && workspace_bytes >= w.bytes, "bm3d: workspace of %lld bytes, need %lld",
                   static_cast<long long>(workspace_bytes), static_cast<long long>(w.bytes));
  if (int rc = require_sm100()) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (a.basic) return run_stage<2>(a, w, a.basic, a.out, a.match2, a.size2, s);
  if (a.stages == B200DN_BM3D_HARD_THRESHOLDING) return run_stage<1>(a, w, nullptr, a.out, a.match1, a.size1, s);
  if (int rc = run_stage<1>(a, w, nullptr, w.basic, a.match1, a.size1, s)) return rc;
  return run_stage<2>(a, w, w.basic, a.out, a.match2, a.size2, s);
}

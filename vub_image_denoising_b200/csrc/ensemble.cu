// ensemble.cu — the data movement of the x8 geometric self-ensemble (b200dn.h, "x8 geometric self-ensemble").
//   dihedral_expand : x [B, C, H, W] -> the 8 flips / rotations, as the even group [4B, C, H, W] and the odd group
//                     [4B, C, W, H] (one read, eight writes)
//   dihedral_reduce : the two groups of network outputs -> [B, C, H, W], each output element the fp32 mean of the 8
//                     positions that hold it, added in k order (eight reads, one write)
// Both are HBM-bound.  A block owns one 32 x 32 tile of one plane.  The flips (even k) map a tile row onto one output
// row, so they go straight from registers; the transposes (odd k) go through a shared-memory tile so that the loads
// and the stores both walk along rows.  With H and W multiples of 4 and 16-byte aligned pointers every access is 128
// bits wide (a reversed row is a reversed sequence of float4 then); otherwise every access is 32 bits wide.
#include "common.cuh"

namespace b200dn {

namespace {

constexpr int DT = 32;              // tile edge
constexpr int DH_THREADS = 256;
constexpr int kMaxTiles = 65535;    // grid y limit: H <= 32 * 65535

// Transform k = 2s + group.  Element x[r][c] of a plane goes to
//   group 0 (k = 0, 2, 4, 6), H x W: row (rows(0, s) ? H-1-r : r), column (cols(0, s) ? W-1-c : c)
//   group 1 (k = 1, 3, 5, 7), W x H: row (cols(1, s) ? W-1-c : c), column (rows(1, s) ? H-1-r : r)
// (torch.rot90 by k % 4 after torch.flip of the columns for k >= 4; tests/test_gpu_ensemble.py holds both kernels
// bit for bit to a torch restatement).
__device__ __forceinline__ bool rows_reversed(int /*group*/, int s) { return s & 1; }
__device__ __forceinline__ bool cols_reversed(int group, int s) {
  return group ? (s == 0 || s == 3) : (s == 1 || s == 2);
}

template <int V>
__device__ __forceinline__ void load(const float* p, bool rev, float (&v)[V]) {
  if constexpr (V == 4) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(p));
    if (rev) v[0] = t.w, v[1] = t.z, v[2] = t.y, v[3] = t.x;
    else     v[0] = t.x, v[1] = t.y, v[2] = t.z, v[3] = t.w;
  } else {
    v[0] = __ldg(p);
  }
}

template <int V>
__device__ __forceinline__ void store(float* p, bool rev, const float (&v)[V]) {
  if constexpr (V == 4) {
    *reinterpret_cast<float4*>(p) = rev ? make_float4(v[3], v[2], v[1], v[0]) : make_float4(v[0], v[1], v[2], v[3]);
  } else {
    *p = v[0];
  }
}

// Thread layout for V-wide accesses along a tile edge: LANES threads per tile row, ROWS rows per pass, PASSES passes.
template <int V>
struct Layout {
  static constexpr int LANES = DT / V, ROWS = DH_THREADS / LANES, PASSES = DT / ROWS;
};

// Group layout: B200DN_DIHEDRAL_INDEX(k, p, planes) is the plane of transform k that holds plane p = b * C + c of x.
// Offset of the V elements of a plane of the even group that hold x[r][c .. c+V) of transform 2s (reversed when
// cols_reversed), and of the odd group's V elements that hold x[r .. r+V)[c] of transform 2s + 1.
template <int V>
__device__ __forceinline__ int64_t even_at(int s, int64_t r, int64_t c, int H, int W) {
  return (rows_reversed(0, s) ? H - 1 - r : r) * W + (cols_reversed(0, s) ? W - V - c : c);
}
template <int V>
__device__ __forceinline__ int64_t odd_at(int s, int64_t r, int64_t c, int H, int W) {
  return (cols_reversed(1, s) ? W - 1 - c : c) * H + (rows_reversed(1, s) ? H - V - r : r);
}

template <int V>
__global__ void __launch_bounds__(DH_THREADS) dihedral_expand_kernel(const float* __restrict__ x, int64_t planes,
                                                                     int H, int W, float* __restrict__ even,
                                                                     float* __restrict__ odd) {
  using L = Layout<V>;
  __shared__ float tile[DT][DT + 1];
  const int t = threadIdx.x;
  const int r0 = blockIdx.y * DT, c0 = blockIdx.x * DT;
  const int64_t hw = static_cast<int64_t>(H) * W;
  for (int64_t p = blockIdx.z; p < planes; p += gridDim.z) {
    const float* src = x + p * hw;
    // row pass: tile row lr, columns lc .. lc+V
    const int lc = (t % L::LANES) * V;
#pragma unroll
    for (int q = 0; q < L::PASSES; ++q) {
      const int lr = t / L::LANES + q * L::ROWS;
      const int r = r0 + lr, c = c0 + lc;
      if (r < H && c < W) {
        float v[V];
        load<V>(src + static_cast<int64_t>(r) * W + c, false, v);
#pragma unroll
        for (int e = 0; e < V; ++e) tile[lr][lc + e] = v[e];
#pragma unroll
        for (int s = 0; s < 4; ++s)
          store<V>(even + B200DN_DIHEDRAL_INDEX(2 * s, p, planes) * hw + even_at<V>(s, r, c, H, W),
                   cols_reversed(0, s), v);
      }
    }
    __syncthreads();
    // column pass: tile column tc, rows tr .. tr+V (one output row of the odd group)
    const int tr = (t % L::LANES) * V;
#pragma unroll
    for (int q = 0; q < L::PASSES; ++q) {
      const int tc = t / L::LANES + q * L::ROWS;
      const int r = r0 + tr, c = c0 + tc;
      if (r < H && c < W) {
        float v[V];
#pragma unroll
        for (int e = 0; e < V; ++e) v[e] = tile[tr + e][tc];
#pragma unroll
        for (int s = 0; s < 4; ++s)
          store<V>(odd + B200DN_DIHEDRAL_INDEX(2 * s + 1, p, planes) * hw + odd_at<V>(s, r, c, H, W),
                   rows_reversed(1, s), v);
      }
    }
    __syncthreads();
  }
}

template <int V>
__global__ void __launch_bounds__(DH_THREADS) dihedral_reduce_kernel(const float* __restrict__ even,
                                                                     const float* __restrict__ odd, int64_t planes,
                                                                     int H, int W, float* __restrict__ out) {
  using L = Layout<V>;
  __shared__ float tile[4][DT][DT + 1];    // the odd transforms' values, in the source's orientation
  const int t = threadIdx.x;
  const int r0 = blockIdx.y * DT, c0 = blockIdx.x * DT;
  const int64_t hw = static_cast<int64_t>(H) * W;
  const int lc = (t % L::LANES) * V, tr = lc;
  for (int64_t p = blockIdx.z; p < planes; p += gridDim.z) {
    // every load of the tile is issued before the first shared-memory store: 8 x PASSES accesses in flight
    float ev[4][L::PASSES][V], od[4][L::PASSES][V];
#pragma unroll
    for (int q = 0; q < L::PASSES; ++q) {
      const int lr = t / L::LANES + q * L::ROWS, tc = lr;
      const int r = r0 + lr, c = c0 + lc;
      if (r < H && c < W) {
#pragma unroll
        for (int s = 0; s < 4; ++s)
          load<V>(even + B200DN_DIHEDRAL_INDEX(2 * s, p, planes) * hw + even_at<V>(s, r, c, H, W),
                  cols_reversed(0, s), ev[s][q]);
      }
      if (r0 + tr < H && c0 + tc < W) {
#pragma unroll
        for (int s = 0; s < 4; ++s)
          load<V>(odd + B200DN_DIHEDRAL_INDEX(2 * s + 1, p, planes) * hw + odd_at<V>(s, r0 + tr, c0 + tc, H, W),
                  rows_reversed(1, s), od[s][q]);
      }
    }
#pragma unroll
    for (int q = 0; q < L::PASSES; ++q) {
      const int tc = t / L::LANES + q * L::ROWS;
      if (r0 + tr < H && c0 + tc < W) {
#pragma unroll
        for (int s = 0; s < 4; ++s)
#pragma unroll
          for (int e = 0; e < V; ++e) tile[s][tr + e][tc] = od[s][q][e];
      }
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < L::PASSES; ++q) {
      const int lr = t / L::LANES + q * L::ROWS;
      const int r = r0 + lr, c = c0 + lc;
      if (r < H && c < W) {
        float v[V];
#pragma unroll
        for (int e = 0; e < V; ++e) {
          float a = ev[0][q][e];                                  // k = 0
#pragma unroll
          for (int s = 0; s < 4; ++s) {
            a = __fadd_rn(a, tile[s][lr][lc + e]);                // k = 2s + 1
            if (s < 3) a = __fadd_rn(a, ev[s + 1][q][e]);         // k = 2s + 2
          }
          v[e] = __fmul_rn(a, 0.125f);
        }
        store<V>(out + p * hw + static_cast<int64_t>(r) * W + c, false, v);
      }
    }
    __syncthreads();
  }
}

bool vec4_ok(int H, int W, const void* a, const void* b, const void* c) {
  return H % 4 == 0 && W % 4 == 0 &&
         ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) | reinterpret_cast<uintptr_t>(c)) & 15) == 0;
}

dim3 dihedral_grid(int64_t planes, int H, int W) {
  return dim3(static_cast<unsigned>(cdiv(W, DT)), static_cast<unsigned>(cdiv(H, DT)),
              static_cast<unsigned>(planes < 65535 ? planes : 65535));
}

}  // namespace
}  // namespace b200dn

extern "C" int b200dn_dihedral_expand(const float* x, int B, int C, int H, int W, float* even, float* odd,
                                      void* stream) {
  using namespace b200dn;
  B200DN_CHECK_ARG(x && even && odd, "dihedral_expand: null pointer");
  B200DN_CHECK_ARG(B > 0 && C > 0 && H > 0 && W > 0, "dihedral_expand: bad shape [%d, %d, %d, %d]", B, C, H, W);
  B200DN_CHECK_ARG(H <= DT * kMaxTiles && W <= DT * kMaxTiles, "dihedral_expand: H, W must be <= %d", DT * kMaxTiles);
  if (int rc = require_sm100()) return rc;
  const int64_t planes = static_cast<int64_t>(B) * C;
  const dim3 grid = dihedral_grid(planes, H, W);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (vec4_ok(H, W, x, even, odd))
    dihedral_expand_kernel<4><<<grid, DH_THREADS, 0, s>>>(x, planes, H, W, even, odd);
  else
    dihedral_expand_kernel<1><<<grid, DH_THREADS, 0, s>>>(x, planes, H, W, even, odd);
  B200DN_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int b200dn_dihedral_reduce(const float* even, const float* odd, int B, int C, int H, int W, float* out,
                                      void* stream) {
  using namespace b200dn;
  B200DN_CHECK_ARG(even && odd && out, "dihedral_reduce: null pointer");
  B200DN_CHECK_ARG(B > 0 && C > 0 && H > 0 && W > 0, "dihedral_reduce: bad shape [%d, %d, %d, %d]", B, C, H, W);
  B200DN_CHECK_ARG(H <= DT * kMaxTiles && W <= DT * kMaxTiles, "dihedral_reduce: H, W must be <= %d", DT * kMaxTiles);
  if (int rc = require_sm100()) return rc;
  const int64_t planes = static_cast<int64_t>(B) * C;
  const dim3 grid = dihedral_grid(planes, H, W);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (vec4_ok(H, W, even, odd, out))
    dihedral_reduce_kernel<4><<<grid, DH_THREADS, 0, s>>>(even, odd, planes, H, W, out);
  else
    dihedral_reduce_kernel<1><<<grid, DH_THREADS, 0, s>>>(even, odd, planes, H, W, out);
  B200DN_CUDA(cudaGetLastError());
  return 0;
}

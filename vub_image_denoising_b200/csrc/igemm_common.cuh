// igemm_common.cuh — pieces shared by the tensor-core convolution kernels:
//   igemm_sm100.cu          per-tap A-tile reload; all modes (3x3, 2x2 stride 2, transposed 2x2, 1x1)
//   conv3x3_slab_sm100.cu   3x3 only; one haloed input slab per 64-channel block, 9 shifted UMMA descriptors (one
//                           CTA per tile, CTA pairs, or a chain of dependent layers in one launch)
// Both write through the same fused epilogue (bias + PReLU + residual + channel-slice store).  The parameter blocks of
// the fused dense block (dense_block_sm100.cu) and the tile walk of the input block (conv_in.cu) live here too.
#pragma once
#include "common.cuh"

#include <cudaTypedefs.h>

namespace b200dn {
namespace igemm {

constexpr int BLOCK_M = 128;  // UMMA M (pixels per accumulator)
constexpr int BLOCK_K = 64;   // 64 x 16-bit = one 128-byte swizzle row
constexpr int A_BYTES = BLOCK_M * BLOCK_K * 2;
constexpr int MAX_N = 256;
constexpr int NUM_THREADS = 256;
constexpr int EPI_THREADS = 128;
constexpr int MAX_STAGES = 8;

struct __align__(64) KParams {
  CUtensorMap tmA0, tmA1, tmW;
  int taps;
  int B, H, W;  // GEMM-M domain (pixels the accumulator rows enumerate)
  int n_cblk, last_k16;
  int cout, block_n;
  int mt;       // A tiles (128 pixels each) sharing one W tile
  int n_tiles_per_group, num_n_tiles;
  int tiles_x, tiles_y, num_tiles;   // spatial tiling in super tiles (mt sub-tiles each)
  int n_pairs, pair_a[3], pair_w[3];
  int wgroups;
  int fmt;  // 1 bf16, 0 fp16
  int num_stages, stage_bytes, tmem_cols;
  // slab kernel only
  int slab_w, slab_bytes, num_slabs;            // slab_bytes = ring slot stride (1 KB multiple)
  int slab_tx;                                  // bytes one slab TMA box delivers
  int wres, n_wplanes;   // weights resident in shared memory (small layers)
  int w_taps;            // filter taps per streamed-W ring stage (1, or 3 = one filter row)
  int cta2, num_m_tiles; // CTA-pair kernel (cta_group::2): two spatial super tiles per W tile, one per CTA
  int epi_staged;        // smem-transposed epilogue with 128-byte-row global stores
  int up_fold;           // transposed conv with 4 * cout <= 256: the four output phases are ONE N tile (A loaded once)
  const float* bias;
  const float* slope;
  int out_kind;
  void* out0;
  void* out1;
  int out_ctot, out_coff;
  const void* res0;
  const void* res1;
  int res_ctot;
  float* out_nchw;
  const float* res_nchw;
  int res_bmod;
  int* sat_flag;         // optional: OR'ed with 1 when an fp16-stored output saturated (|v| >= 65504) or was NaN
#ifdef B200DN_TIMELINE
  unsigned long long* tl;   // diagnostics build only: 16 %globaltimer slots of this launch (CTA 0), see TL_MARK
#endif
};

// Launch timeline (diagnostics build, -DB200DN_TIMELINE; tools/launch_timeline.py): CTA 0 of every tensor-core launch
// stores %globaltimer at fixed points, so the hand-off between dependent launches of a small-batch forward (exit of
// launch n -> entry / griddepcontrol.wait return / first MMA / first drained accumulator of launch n + 1) can be read
// on one clock.  Compiled out of the product library.
enum { TL_ENTRY = 0, TL_SETUP = 1, TL_DEP = 2, TL_MMA0 = 3, TL_MMA_END = 4, TL_ACC0 = 5, TL_EPI_END = 6, TL_EXIT = 7, TL_SM = 8 };
#ifdef B200DN_TIMELINE
__device__ __forceinline__ unsigned long long tl_now() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
#define TL_MARK(p, slot)                                          \
  do {                                                            \
    if ((p).tl != nullptr && blockIdx.x == 0) (p).tl[slot] = tl_now(); \
  } while (0)
#define TL_MARK_ONCE(p, slot, flag)                               \
  do {                                                            \
    if (!(flag)) {                                                \
      (flag) = true;                                              \
      TL_MARK(p, slot);                                           \
    }                                                             \
  } while (0)
#else
#define TL_MARK(p, slot) do {} while (0)
#define TL_MARK_ONCE(p, slot, flag) do {} while (0)
#endif

struct TileCoord {
  int b, y0, x0, grp, n0;
};

// tile -> (image, super-tile origin, N group, N offset); super tile = tile_w x tile_h pixels
__device__ __forceinline__ TileCoord decode_tile(int tile, int num_n_tiles, int n_tiles_per_group, int block_n,
                                                 int tiles_x, int tiles_y, int tile_w, int tile_h) {
  TileCoord t;
  const int m_tile = tile / num_n_tiles;
  const int nt = tile - m_tile * num_n_tiles;
  t.grp = nt / n_tiles_per_group;
  t.n0 = (nt - t.grp * n_tiles_per_group) * block_n;
  const int per_img = tiles_x * tiles_y;
  t.b = m_tile / per_img;
  const int r = m_tile - t.b * per_img;
  const int ty = r / tiles_x;
  t.y0 = ty * tile_h;
  t.x0 = (r - ty * tiles_x) * tile_w;
  return t;
}

// Division-free walk over the tiles blockIdx.x, blockIdx.x + grid, ... of a conv3x3 layer (one N group): the stride
// `grid` is decomposed ONCE into mixed-radix digits (N tile, tile column, tile row, image) and added with carries per
// step.  decode_tile costs four integer divisions (~110 SASS instructions with long dependent chains) per tile and warp;
// on the small-N layers the epilogue warps that execute it are what the MMA issuers wait for (ncu: issuer warps stalled
// on the accumulator-empty barrier, profiles/r02_base_conv_32_16_summary.txt).
struct TileWalker {
  int nt, tx, ty, b;          // current digits
  int s_nt, s_tx, s_ty, s_b;  // digits of the stride
  int num_n_tiles, tiles_x, tiles_y;
  __device__ __forceinline__ void init(int tile, int stride, int num_n_tiles_, int tiles_x_, int tiles_y_) {
    num_n_tiles = num_n_tiles_, tiles_x = tiles_x_, tiles_y = tiles_y_;
    int m = tile / num_n_tiles;
    nt = tile - m * num_n_tiles;
    int q = m / tiles_x;
    tx = m - q * tiles_x;
    b = q / tiles_y;
    ty = q - b * tiles_y;
    m = stride / num_n_tiles;
    s_nt = stride - m * num_n_tiles;
    q = m / tiles_x;
    s_tx = m - q * tiles_x;
    s_b = q / tiles_y;
    s_ty = q - s_b * tiles_y;
  }
  __device__ __forceinline__ void next() {
    nt += s_nt;
    int c = nt >= num_n_tiles ? 1 : 0;
    nt -= c ? num_n_tiles : 0;
    tx += s_tx + c;
    c = tx >= tiles_x ? 1 : 0;
    tx -= c ? tiles_x : 0;
    ty += s_ty + c;
    c = ty >= tiles_y ? 1 : 0;
    ty -= c ? tiles_y : 0;
    b += s_b + c;
  }
  __device__ __forceinline__ TileCoord coord(int block_n, int tile_w, int tile_h) const {
    TileCoord t;
    t.b = b, t.y0 = ty * tile_h, t.x0 = tx * tile_w, t.grp = 0, t.n0 = nt * block_n;
    return t;
  }
  // with N groups (the four phases of the transposed conv): nt = grp * n_tiles_per_group + n tile
  __device__ __forceinline__ TileCoord coord_groups(int block_n, int n_tiles_per_group, int tile_w, int tile_h) const {
    TileCoord t;
    t.b = b, t.y0 = ty * tile_h, t.x0 = tx * tile_w;
    if (n_tiles_per_group == 1) {
      t.grp = nt, t.n0 = 0;
    } else {
      t.grp = nt / n_tiles_per_group;
      t.n0 = (nt - t.grp * n_tiles_per_group) * block_n;
    }
    return t;
  }
};

template <bool kBf16>
__device__ __forceinline__ float cvt_lo(uint32_t v) {
  return kBf16 ? bf16_lo(v) : f16_lo(v);
}
template <bool kBf16>
__device__ __forceinline__ float cvt_hi(uint32_t v) {
  return kBf16 ? bf16_hi(v) : f16_hi(v);
}
template <bool kBf16>
__device__ __forceinline__ uint32_t pack2(float a, float b) {
  if (kBf16) return pack_bf16x2(a, b);
  // fp16 storage saturates instead of overflowing to inf: one F2FP.SATFINITE instead of four FMNMX + F2FP
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return r;
}

// fp16 saturation watch: running per-half maximum of |v| over the packed fp16 pairs a thread stores (NaN propagates);
// one atomicOr per thread at most, and only if something saturated.
__device__ __forceinline__ uint32_t sat_track(uint32_t m, uint32_t h) {
  uint32_t r;
  asm("{\n\t.reg .b32 a;\n\tabs.f16x2 a, %2;\n\tmax.NaN.f16x2 %0, %1, a;\n\t}" : "=r"(r) : "r"(m), "r"(h));
  return r;
}
__device__ __forceinline__ void sat_report(int* flag, uint32_t m) {
  if (flag != nullptr && (((m & 0x7fffu) >= 0x7bffu) || ((m >> 16) >= 0x7bffu))) atomicOr(flag, 1);
}

struct EpiArgs {
  void* out0;
  void* out1;
  const void* res0;
  const void* res1;
  int out_ctot, out_coff, res_ctot, cout;
  int out_kind, is_bf16;
  float* out_nchw;
  const float* res_nchw;
  int res_bmod, H, W;
  int* sat_flag;
};

__device__ __forceinline__ EpiArgs make_epi_args(const KParams& p) {
  EpiArgs e;
  e.out0 = p.out0, e.out1 = p.out1, e.res0 = p.res0, e.res1 = p.res1;
  e.out_ctot = p.out_ctot, e.out_coff = p.out_coff, e.res_ctot = p.res_ctot, e.cout = p.cout;
  e.out_kind = p.out_kind, e.is_bf16 = p.fmt != 0;
  e.out_nchw = p.out_nchw, e.res_nchw = p.res_nchw, e.res_bmod = p.res_bmod, e.H = p.H, e.W = p.W;
  e.sat_flag = p.fmt != 0 ? nullptr : p.sat_flag;   // bf16 storage has fp32's exponent range: nothing to watch
  return e;
}

// 16 accumulator columns of one pixel -> 16 channels of the NHWC slice.
template <bool kBf16>
__device__ __forceinline__ void epilogue_nhwc16(const EpiArgs& e, float (&v)[16], int64_t out_pix, int64_t res_pix,
                                                int ch0, uint32_t& satm) {
  if (ch0 >= e.cout) return;
  const bool half1 = (ch0 + 8) < e.cout;  // second 8-channel group inside cout
  if (e.res0 != nullptr) {
    const uint4* r0 = reinterpret_cast<const uint4*>(static_cast<const uint16_t*>(e.res0) + res_pix * e.res_ctot + ch0);
    uint4 q[2];
    q[0] = __ldg(r0);
    q[1] = half1 ? __ldg(r0 + 1) : make_uint4(0, 0, 0, 0);
    const uint32_t* w = reinterpret_cast<const uint32_t*>(q);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      v[2 * j] += cvt_lo<kBf16>(w[j]);
      v[2 * j + 1] += cvt_hi<kBf16>(w[j]);
    }
    if (e.res1 != nullptr) {
      const uint4* r1 =
          reinterpret_cast<const uint4*>(static_cast<const uint16_t*>(e.res1) + res_pix * e.res_ctot + ch0);
      q[0] = __ldg(r1);
      q[1] = half1 ? __ldg(r1 + 1) : make_uint4(0, 0, 0, 0);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        v[2 * j] += cvt_lo<kBf16>(w[j]);
        v[2 * j + 1] += cvt_hi<kBf16>(w[j]);
      }
    }
  }
  uint32_t hi[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) hi[j] = pack2<kBf16>(v[2 * j], v[2 * j + 1]);
  if (!kBf16 && e.sat_flag != nullptr) {
#pragma unroll
    for (int j = 0; j < 8; ++j) satm = sat_track(satm, hi[j]);
  }
  uint4* o0 = reinterpret_cast<uint4*>(static_cast<uint16_t*>(e.out0) + out_pix * e.out_ctot + e.out_coff + ch0);
  o0[0] = make_uint4(hi[0], hi[1], hi[2], hi[3]);
  if (half1) o0[1] = make_uint4(hi[4], hi[5], hi[6], hi[7]);
  if (e.out1 != nullptr) {
    uint32_t lo[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float a = v[2 * j] - cvt_lo<kBf16>(hi[j]);
      const float b = v[2 * j + 1] - cvt_hi<kBf16>(hi[j]);
      lo[j] = pack2<kBf16>(a, b);
    }
    uint4* o1 = reinterpret_cast<uint4*>(static_cast<uint16_t*>(e.out1) + out_pix * e.out_ctot + e.out_coff + ch0);
    o1[0] = make_uint4(lo[0], lo[1], lo[2], lo[3]);
    if (half1) o1[1] = make_uint4(lo[4], lo[5], lo[6], lo[7]);
  }
}

// Drain one 128 x block_n accumulator (this thread = one pixel row): TMEM -> +bias -> PReLU -> (+residual) -> store.
// `release_bar` != 0: arrive on it right after the last TMEM read (hands the accumulator stage back to the MMA warps).
__device__ __forceinline__ void epilogue_subtile(const EpiArgs& e, uint32_t taddr, int block_n, const float* bs,
                                                 const float* ss, bool valid, int b, int y, int x, int64_t out_pix,
                                                 int64_t res_pix, int n0, uint32_t release_bar, uint32_t& satm,
                                                 bool cluster_rel = false) {
  for (int c0 = 0; c0 < block_n; c0 += 16) {
    uint32_t r[16];
    tmem_ld16(taddr + c0, r);
    tmem_ld_wait();
    if (release_bar != 0 && c0 + 16 >= block_n) {
      tc_fence_before();
      // one arrive per WARP (the barrier counts warps): 128-256 per-thread arrives on one shared-memory word serialise
      // and sit on the path that hands the accumulator stage back to the MMA issuers
      __syncwarp();
      if ((threadIdx.x & 31) == 0) {
        if (cluster_rel)
          mbar_arrive_cluster(release_bar);   // CTA pair: the barrier lives in the leader CTA
        else
          mbar_arrive(release_bar);
      }
    }
    if (!valid) continue;
    float v[16];
    const float4* b4 = reinterpret_cast<const float4*>(bs + c0);
    const float4* s4 = reinterpret_cast<const float4*>(ss + c0);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float4 bb = b4[q];
      const float4 sl = s4[q];
      float a;
      a = __uint_as_float(r[4 * q + 0]) + bb.x;
      v[4 * q + 0] = a > 0.f ? a : a * sl.x;
      a = __uint_as_float(r[4 * q + 1]) + bb.y;
      v[4 * q + 1] = a > 0.f ? a : a * sl.y;
      a = __uint_as_float(r[4 * q + 2]) + bb.z;
      v[4 * q + 2] = a > 0.f ? a : a * sl.z;
      a = __uint_as_float(r[4 * q + 3]) + bb.w;
      v[4 * q + 3] = a > 0.f ? a : a * sl.w;
    }
    if (e.out_kind == B200DN_OUT_NHWC16) {
      if (e.is_bf16)
        epilogue_nhwc16<true>(e, v, out_pix, res_pix, n0 + c0, satm);
      else
        epilogue_nhwc16<false>(e, v, out_pix, res_pix, n0 + c0, satm);
    } else {
      // fp32 NCHW output block: prelu(conv) + inputs   (UNet/RDUNet_model.py:186)
      const int64_t hw = static_cast<int64_t>(e.H) * e.W;
      const int64_t sp = static_cast<int64_t>(y) * e.W + x;
#pragma unroll
      for (int jj = 0; jj < 16; ++jj) {
        const int c = n0 + c0 + jj;
        if (c < e.cout) {
          float o = v[jj];
          if (e.res_nchw != nullptr)
            o += __ldg(e.res_nchw + (static_cast<int64_t>(b % e.res_bmod) * e.cout + c) * hw + sp);
          e.out_nchw[(static_cast<int64_t>(b) * e.cout + c) * hw + sp] = o;
        }
      }
    }
  }
}

// ---- staged epilogue -------------------------------------------------------------------------------------
// The direct epilogue above has every thread store 16 B of its own pixel: 32 different 128-byte lines per
// warp instruction (32 L1 wavefronts for 512 useful bytes).  The staged variant transposes a [32 pixel x 64
// channel] block through a per-warp 4 KB shared-memory buffer (16-byte chunks XOR-swizzled by the row, so both
// the row-wise writes and the 4-rows-per-instruction reads are bank-conflict free) and then stores / loads whole
// 128-byte pixel rows: 8 lanes per pixel, 4 pixels per warp instruction.  Single-plane formats, cout % 64 == 0.
struct RowMap {
  int b, y0, x0;       // image, tile origin (for the sub-tile)
  int tw_shift;        // log2 of the accumulator tile width in pixels (4: tap kernel, 3: slab kernel)
  int H, W;            // GEMM-M domain
  int up, ky, kx;      // transposed conv: output pixel = (2y+ky, 2x+kx) in a 2H x 2W image
};

__device__ __forceinline__ bool row_pixels(const RowMap& m, int row, int64_t& out_pix, int64_t& res_pix) {
  const int th = row >> m.tw_shift, tw = row & ((1 << m.tw_shift) - 1);
  const int y = m.y0 + th, x = m.x0 + tw;
  res_pix = (static_cast<int64_t>(m.b) * m.H + y) * m.W + x;
  out_pix = m.up ? (static_cast<int64_t>(m.b) * (2 * m.H) + (2 * y + m.ky)) * (2 * m.W) + (2 * x + m.kx) : res_pix;
  return (y < m.H) && (x < m.W);
}

__device__ __forceinline__ void epilogue_subtile_staged(const EpiArgs& e, uint32_t taddr, int block_n, const float* bs,
                                                        const float* ss, const RowMap& m, int row0, int lane, int n0,
                                                        uint32_t release_bar, uint8_t* stg, uint32_t& satm,
                                                        bool cluster_rel = false) {
  const uint32_t my_row = static_cast<uint32_t>(lane);
  const int sub_row = lane >> 3, chunk = lane & 7;   // coalesced phases: 4 rows x 8 chunks per instruction
  // per-lane addresses of its 8 coalesced rows (invariant over the channel groups of this sub-tile)
  uint16_t* optr[8];
  const uint16_t* rptr[8];
  uint32_t okmask = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    int64_t op, rp;
    const bool ok = row_pixels(m, row0 + i * 4 + sub_row, op, rp);
    okmask |= (ok ? 1u : 0u) << i;
    optr[i] = static_cast<uint16_t*>(e.out0) + op * e.out_ctot + e.out_coff + n0 + chunk * 8;
    rptr[i] = static_cast<const uint16_t*>(e.res0) + rp * e.res_ctot + n0 + chunk * 8;
  }
  // staging offsets of those rows, and of this thread's own row (compute phase)
  const uint32_t co_off = static_cast<uint32_t>(sub_row * 128 + ((chunk ^ sub_row) << 4));   // + i*512, XOR fixed below
  (void)co_off;
  for (int c0 = 0; c0 < block_n; c0 += 64) {
    if (e.res0 != nullptr) {
      // residual tile -> staging (coalesced 128-byte rows)
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int r = i * 4 + sub_row;
        uint4 q = make_uint4(0, 0, 0, 0);
        if ((okmask >> i) & 1u) q = __ldg(reinterpret_cast<const uint4*>(rptr[i] + c0));
        *reinterpret_cast<uint4*>(stg + r * 128 + ((chunk ^ (r & 7)) << 4)) = q;
      }
      __syncwarp();
    }
#pragma unroll
    for (int q4 = 0; q4 < 4; ++q4) {
      uint32_t r[16];
      tmem_ld16(taddr + c0 + 16 * q4, r);
      tmem_ld_wait();
      if (release_bar != 0 && c0 + 64 >= block_n && q4 == 3) {
        tc_fence_before();
        __syncwarp();
        if ((threadIdx.x & 31) == 0) {
          if (cluster_rel)
            mbar_arrive_cluster(release_bar);
          else
            mbar_arrive(release_bar);
        }
      }
      float v[16];
      const float4* b4 = reinterpret_cast<const float4*>(bs + c0 + 16 * q4);
      const float4* s4 = reinterpret_cast<const float4*>(ss + c0 + 16 * q4);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float4 bb = b4[q];
        const float4 sl = s4[q];
        float a;
        a = __uint_as_float(r[4 * q + 0]) + bb.x;
        v[4 * q + 0] = a > 0.f ? a : a * sl.x;
        a = __uint_as_float(r[4 * q + 1]) + bb.y;
        v[4 * q + 1] = a > 0.f ? a : a * sl.y;
        a = __uint_as_float(r[4 * q + 2]) + bb.z;
        v[4 * q + 2] = a > 0.f ? a : a * sl.z;
        a = __uint_as_float(r[4 * q + 3]) + bb.w;
        v[4 * q + 3] = a > 0.f ? a : a * sl.w;
      }
      uint4* s0 = reinterpret_cast<uint4*>(stg + my_row * 128 + (((2 * q4) ^ (my_row & 7)) << 4));
      uint4* s1 = reinterpret_cast<uint4*>(stg + my_row * 128 + (((2 * q4 + 1) ^ (my_row & 7)) << 4));
      if (e.res0 != nullptr) {
        const uint4 ra = *s0, rb = *s1;
        const uint32_t w[8] = {ra.x, ra.y, ra.z, ra.w, rb.x, rb.y, rb.z, rb.w};
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          v[2 * j] += e.is_bf16 ? bf16_lo(w[j]) : f16_lo(w[j]);
          v[2 * j + 1] += e.is_bf16 ? bf16_hi(w[j]) : f16_hi(w[j]);
        }
      }
      uint32_t h[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) h[j] = e.is_bf16 ? pack2<true>(v[2 * j], v[2 * j + 1]) : pack2<false>(v[2 * j], v[2 * j + 1]);
      if (e.sat_flag != nullptr) {   // only set for fp16 storage
#pragma unroll
        for (int j = 0; j < 8; ++j) satm = sat_track(satm, h[j]);
      }
      *s0 = make_uint4(h[0], h[1], h[2], h[3]);
      *s1 = make_uint4(h[4], h[5], h[6], h[7]);
    }
    __syncwarp();
    // staging -> global: whole 128-byte pixel rows
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int r = i * 4 + sub_row;
      const uint4 q = *reinterpret_cast<const uint4*>(stg + r * 128 + ((chunk ^ (r & 7)) << 4));
      if ((okmask >> i) & 1u) *reinterpret_cast<uint4*>(optr[i] + c0) = q;
    }
    __syncwarp();
  }
}

// stage the tile's bias / PReLU slopes in shared memory (called by the 128 epilogue threads)
__device__ __forceinline__ void stage_bias_slope(float* bs, float* ss, const float* bias, const float* slope, int n0,
                                                 int block_n, int cout, int et, int n_threads = EPI_THREADS) {
  for (int i = et; i < block_n; i += n_threads) {
    const int c = n0 + i;
    bs[i] = (c < cout) ? __ldg(bias + c) : 0.f;
    ss[i] = (slope != nullptr && c < cout) ? __ldg(slope + c) : 1.f;
  }
  asm volatile("bar.sync 1, %0;" ::"r"(n_threads) : "memory");
}

// NK consecutive k16 steps of one filter tap: D (+)= A[128 x 16] * B[N x 16]^T, descriptors advanced by 32 B (2 units).
// Compile-time NK keeps the single-thread issue loop straight-line (3 SASS instructions per UMMA); ncu had shown the
// issuer warp, not the data, limiting the small-N layers.
template <int NK, bool CTA2>
__device__ __forceinline__ void issue_k16_steps(uint32_t d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                                uint32_t accumulate) {
#pragma unroll
  for (int k = 0; k < NK; ++k) {
    if (CTA2)
      umma_f16_2cta(d, adesc + 2 * k, bdesc + 2 * k, idesc, k == 0 ? accumulate : 1u);
    else
      umma_f16(d, adesc + 2 * k, bdesc + 2 * k, idesc, k == 0 ? accumulate : 1u);
  }
}
// Streamed-W ring cursor of an MMA issuer: barrier addresses and the B descriptor advance together.
struct WRing {
  uint32_t full, empty, phase;
  uint64_t desc;
  uint32_t full0, empty0, full_end;
  uint64_t desc0, step;
  __device__ __forceinline__ void advance() {
    full += 8, empty += 8, desc += step;
    if (full == full_end) {
      full = full0, empty = empty0, desc = desc0;
      phase ^= 1u;
    }
  }
};

// The 9 taps of one 64-channel block of a slab, weights streamed through the ring.  WT = taps per ring stage:
//   WT = 1: per tap wait for the W tile, issue NK UMMAs, commit the stage back to the W producer;
//   WT = 3: one stage holds the three taps of a filter row (tiles `tap_step` apart), so the barrier wait, the commit
//           and the ring bookkeeping are paid once per 3 taps — for N <= 64 (UMMAs of <= 32 clk) the issuer warp,
//           not the tensor pipe, is what those instructions delay.
// `arow` = descriptor of the slab row of tap (0, 0).
template <int NK, bool CTA2, int WT>
__device__ __forceinline__ void issue_slab_block_streamed(uint32_t d, uint64_t arow, uint64_t row_step, WRing& w,
                                                          uint64_t tap_step, uint32_t idesc, uint32_t& accumulate) {
#pragma unroll 1
  for (int dy = 0; dy < 3; ++dy, arow += row_step) {
    if (WT == 3) {
      mbar_wait(w.full, w.phase);
      tc_fence_after();
      if (elect_one()) {
        uint64_t bdesc = w.desc;
#pragma unroll
        for (int dx = 0; dx < 3; ++dx, bdesc += tap_step) {
          issue_k16_steps<NK, CTA2>(d, arow + static_cast<uint64_t>(dx * 8), bdesc, idesc, dx == 0 ? accumulate : 1u);
        }
        if (CTA2)
          umma_commit_2cta(w.empty, 3);
        else
          umma_commit(w.empty);
      }
      __syncwarp();
      accumulate = 1;
      w.advance();
    } else {
#pragma unroll
      for (int dx = 0; dx < 3; ++dx) {
        mbar_wait(w.full, w.phase);
        tc_fence_after();
        if (elect_one()) {
          issue_k16_steps<NK, CTA2>(d, arow + static_cast<uint64_t>(dx * 8), w.desc, idesc, accumulate);
          if (CTA2)
            umma_commit_2cta(w.empty, 3);
          else
            umma_commit(w.empty);
        }
        __syncwarp();
        accumulate = 1;
        w.advance();
      }
    }
  }
}
template <bool CTA2>
__device__ __forceinline__ void issue_slab_block_streamed_n(int nk, int wt, uint32_t d, uint64_t arow, uint64_t row_step,
                                                            WRing& w, uint64_t tap_step, uint32_t idesc,
                                                            uint32_t& accumulate) {
  // one dispatch per 9 taps; inside, the k16 count and the stage shape are compile-time constants
  if (wt == 3) {
    switch (nk) {
      case 4: issue_slab_block_streamed<4, CTA2, 3>(d, arow, row_step, w, tap_step, idesc, accumulate); break;
      case 3: issue_slab_block_streamed<3, CTA2, 3>(d, arow, row_step, w, tap_step, idesc, accumulate); break;
      case 2: issue_slab_block_streamed<2, CTA2, 3>(d, arow, row_step, w, tap_step, idesc, accumulate); break;
      default: issue_slab_block_streamed<1, CTA2, 3>(d, arow, row_step, w, tap_step, idesc, accumulate); break;
    }
  } else {
    switch (nk) {
      case 4: issue_slab_block_streamed<4, CTA2, 1>(d, arow, row_step, w, tap_step, idesc, accumulate); break;
      case 3: issue_slab_block_streamed<3, CTA2, 1>(d, arow, row_step, w, tap_step, idesc, accumulate); break;
      case 2: issue_slab_block_streamed<2, CTA2, 1>(d, arow, row_step, w, tap_step, idesc, accumulate); break;
      default: issue_slab_block_streamed<1, CTA2, 1>(d, arow, row_step, w, tap_step, idesc, accumulate); break;
    }
  }
}
// Same with the weights resident in shared memory ([tap][N x 64] tiles `bstep` apart); called by ONE elected thread.
template <int NK>
__device__ __forceinline__ void issue_slab_block_resident(uint32_t d, uint64_t arow, uint64_t row_step, uint64_t bdesc,
                                                          uint64_t bstep, uint32_t idesc, uint32_t accumulate) {
#pragma unroll 1
  for (int dy = 0; dy < 3; ++dy, arow += row_step) {
#pragma unroll
    for (int dx = 0; dx < 3; ++dx, bdesc += bstep) {
      issue_k16_steps<NK, false>(d, arow + static_cast<uint64_t>(dx * 8), bdesc, idesc, accumulate);
      accumulate = 1;
    }
  }
}

// parameter block of the fused dense-block kernel (dense_block_sm100.cu)
struct __align__(64) FusedParams {
  CUtensorMap tmX;
  CUtensorMap tmW[4];
  int B, H, W;
  int regions_x, regions_y, num_regions;
  int fmt;                       // 1 bf16, 0 fp16
  const float* bias[4];
  const float* slope[4];
  const void* in;                // block input (NHWC 16-bit, channels [0, 32)): TMA source and the `+ x` residual
  int in_ctot;
  void* out;
  int out_ctot, out_coff;
  int* sat_flag;
  // bias / PReLU slopes by accumulator column [o0 | o1 | o2 | o3] as VALUES in the launch parameters (constant bank): the
  // epilogue then reads them as instruction operands instead of broadcast LDS (11 % of the kernel's shared-memory
  // wavefronts).  Filled by b200dn_dense_block_set_epilogue_constants; epi_const = 0: staged in shared memory from bias[] / slope[]
  float cbias[80], cslope[80];
  int epi_const;
  long long* dbg;                // optional timeline buffer (tools/dense_block_timeline.py): CTA 0 logs (event, clock64)
#ifdef B200DN_TIMELINE
  unsigned long long* tl;        // diagnostics build only: the launch-timeline slots (TL_MARK)
#endif
};

// parameter block of the multi-layer chain kernel (conv3x3_slab_sm100.cu): the layers' own parameter blocks (ring
// geometry unified by the host) + the work list and the inter-tile dependency counters
constexpr int CHAIN_MAX_LAYERS = 4;
struct __align__(64) ChainParams {
  KParams L[CHAIN_MAX_LAYERS];
  int n_layers;
  int item_base[CHAIN_MAX_LAYERS + 1];   // first work item (pair tile) of each layer, layer-major
  int flag_need[CHAIN_MAX_LAYERS];       // arrivals per launch that complete a spatial tile of layer l
  int nmax;                              // TMEM columns between accumulators (largest N of the chain)
  int tmem_cols;
  uint32_t* flags;                       // [n_layers - 1][num_m_tiles] monotonic arrival counters
  uint32_t* sync;                        // [0] launches completed, [1] CTAs that left the current launch
};

// A fully resolved launch: kernel variant, launch geometry and the parameter block (with its encoded tensor maps).
// b200dn_igemm builds one per call; b200dn_igemm_prepare keeps it, so that later launches cost one cudaLaunchKernelExC.
struct LaunchCfg {
  KParams p;          // kind 0: the per-layer implicit-GEMM kernels
  FusedParams f;      // kind 1: the fused dense block
  ChainParams c;      // kind 2: several dependent 3x3 layers in one launch
  int kind;
  const void* kernel;
  int grid, threads, smem, cluster;
  int cooperative;    // all CTAs must be co-resident (kind 2)
  const void* alt_kernel;   // kind 1: the kernel variant that takes bias / slopes from the launch parameters
};
#ifdef B200DN_TIMELINE
// 16 device slots for the next configured launch, labelled for the dump (igemm_sm100.cu)
unsigned long long* timeline_slots(const char* label);
#endif
using PFN_encodeTiled = PFN_cuTensorMapEncodeTiled;
// the driver's cuTensorMapEncodeTiled entry point (igemm_sm100.cu); 0 on success
int get_tensor_map_encoder(PFN_encodeTiled* fn);
// fused dense block (dense_block_sm100.cu): validate, encode, resolve
int configure_dense_block(const b200dn_dense_block_args& a, LaunchCfg* cfg, PFN_encodeTiled encode_fn);
// chain of dependent 3x3 layers (conv3x3_slab_sm100.cu): B200DN_E_UNSUP when the layers do not qualify
size_t conv_chain_workspace_bytes(const b200dn_igemm_args* layers, int n);
int configure_conv_chain(const b200dn_igemm_args* layers, int n, void* workspace, int flags, LaunchCfg* cfg);
// slab-kernel resolver (conv3x3_slab_sm100.cu); cfg->p is fully populated by igemm_configure.  Picks the template
// variant and opts it in to its dynamic shared memory on the current device.
int resolve_conv3x3_slab(LaunchCfg* cfg, int grid);
// CTA-pair variant (conv3x3_slab_sm100.cu); grid = 2 x clusters
int resolve_conv3x3_slab2(LaunchCfg* cfg, int grid);
// shared-memory budget of the slab kernel, used by the host to size the rings
constexpr int SLAB_DATA_BYTES = 200 * 1024;   // slab + W rings when the staged epilogue is in use
constexpr int EPI_STAGING_BYTES = 16 * 1024;  // 4 epilogue warps x [32 rows x 128 B]
constexpr int SLAB_WRES_BYTES = SLAB_DATA_BYTES + EPI_STAGING_BYTES;   // resident-weight layers (cout < 64) use both
constexpr int SLAB_MAX_SLABS = 6;              // slab ring depth limit (barrier map has room for 8)
constexpr int SLAB_CTRL_BYTES = 384;           // mbarriers + TMEM pointer, ahead of the staged bias / slopes
constexpr int SLAB_TILE_W = 8;    // output tile: 8 wide x 16 tall pixels per accumulator
constexpr int SLAB_TILE_H = 16;

}  // namespace igemm

// igemm_sm100.cu: validate `a`, choose kernel family / tiling / ring sizes, encode the tensor maps into `cfg`
int igemm_configure(const b200dn_igemm_args& a, igemm::LaunchCfg* cfg, b200dn_igemm_plan_info* info = nullptr,
                    int sms_override = 0);
}  // namespace b200dn

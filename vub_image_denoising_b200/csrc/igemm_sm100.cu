// igemm_sm100.cu — the tcgen05/TMEM implicit-GEMM convolution of the RDUNet hot path.
//
// One persistent, warp-specialised kernel covers every GEMM-shaped layer of the network
// (reference: UNet/RDUNet_model.py:49-115, diffusion_denoising/Unet/Unet_model.py:23-89):
//
//   CONV3X3  D[pix, co] = sum_{tap,ci} X[pix + (dy,dx), ci] * W[tap][co][ci]       (zero pad 1)
//   DOWN2X2  D[opix, co] = sum_{ky,kx,ci} X[2*opix + (ky,kx), ci] * W[tap][co][ci]
//   UP2X2    D[pix, (ky,kx,co)] = sum_ci X[pix, ci] * Wt[ky*2+kx][co][ci]  -> scattered to (2y+ky, 2x+kx)
//
// Layout: activations NHWC 16-bit (bf16 or fp16), one or two planes (hi, lo); a layer reads the channel
// prefix [0,cin) of its input buffer and writes the channel slice [coff, coff+cout) of its output buffer,
// so the dense-block concatenations of the reference never materialise.
//
// Pipeline per CTA (256 threads, 1 CTA/SM, grid = #SMs, static round-robin tile schedule):
//   warp 0 / lane 0 : TMA producer.  Per K step (pair, tap, 64-channel block) one haloed A box
//                     [8 x 16 pixels x 64 ch] (OOB zero fill == conv padding) and one W box [N x 64] land
//                     in a 128B-swizzled smem ring stage and complete on its mbarrier.
//   warp 1 / lane 0 : MMA issuer.  tcgen05.mma.cta_group::1.kind::f16, M=128, N=block_n, K=16, fp32
//                     accumulator in TMEM (2 accumulator stages so the epilogue overlaps the next tile).
//   warp 2          : TMEM allocator.
//   warps 4..7      : epilogue.  tcgen05.ld -> +bias -> PReLU -> (+residual) -> 16-bit planes into the
//                     NHWC channel slice, or fp32 NCHW (+fp32 NCHW residual) for the output block.
#include "igemm_common.cuh"
#ifdef B200DN_TIMELINE
#include <mutex>
#include <string>
#include <vector>
#endif

#include <mutex>
#include <new>
#include <stdlib.h>
#include <string.h>

#ifndef B200DN_DEFAULT_CONV3X3_IMPL
#define B200DN_DEFAULT_CONV3X3_IMPL 2
#endif

namespace b200dn {

using namespace igemm;

namespace {

constexpr int TILE_W = 16;   // accumulator tile of the tap-reload kernel: 16 wide x 8 tall pixels
constexpr int TILE_H = 8;
constexpr int RING_BYTES = 176 * 1024;
constexpr int TAP_STAGING_BYTES = 32 * 1024;                 // up to 8 epilogue warps x [32 rows x 128 B]
constexpr int DATA_BYTES = RING_BYTES + TAP_STAGING_BYTES;   // [A/W ring | epilogue staging]
constexpr int SMEM_BYTES = 1024 + DATA_BYTES + 256 + 2 * 2 * MAX_N * 4;

// MODE: 0 = CONV3X3 (9 taps, shifted 4-D boxes), 1 = DOWN2X2 (4 taps, 5-D map), 2 = UP2X2 / CONV1X1 (one tap)
// MT:   A tiles (128 pixels each, x-adjacent) per W tile and pipeline stage.
//
// Warp roles (256 threads): 0 = A-tile TMA producer, 2 = TMEM allocator then W-tile TMA producer,
// 1 = MMA issuer of sub-tile 0, 3 = MMA issuer of sub-tile 1 (MT == 2), 4..7 = epilogue.
// ncu showed the single-thread issue loops (uniform-datapath instructions at ~5 cycles each), not the
// tensor pipe, TMA or L2, bound the first version of this kernel (profiles/r01_igemm_v1_n64.txt); hence
// two producers, two issuers with independent accumulators, and branch-free inner paths.
// The transposed conv (MODE 2, one accumulator, N = 256) has a short K loop (K = Cin) and a 256-column epilogue:
// ncu/event timing showed it epilogue-bound, so that variant runs TWO epilogue warp groups (hardware warps 0-3 and
// 8-11), each draining half of the accumulator's columns.  (For the 3x3 kernels extra epilogue warps were measured
// to be slower: they take issue slots from the MMA issue loops.)
template <int MODE, int MT>
constexpr int epi_groups() { return (MODE == 2 && MT == 1) ? 2 : 1; }

template <int MODE, int MT>
__global__ void __launch_bounds__(NUM_THREADS + EPI_THREADS * (epi_groups<MODE, MT>() - 1), 1)
igemm_kernel(const __grid_constant__ KParams p) {
  constexpr int EG = epi_groups<MODE, MT>();
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_u32 = smem_u32(smem_raw);
  const uint32_t smem_base = (raw_u32 + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - raw_u32);
  const uint32_t bars = smem_base + DATA_BYTES;
  if (threadIdx.x == 0) TL_MARK(p, TL_ENTRY);
  // barrier map: full[8] @0, empty[8] @64, tmem_full[2] @128, tmem_empty[2] @144, tmem ptr @160
  uint32_t* tmem_ptr_s = reinterpret_cast<uint32_t*>(smem_gen + DATA_BYTES + 160);
  float* epi_bias = reinterpret_cast<float*>(smem_gen + DATA_BYTES + 256);  // [2][MAX_N]
  float* epi_slope = epi_bias + 2 * MAX_N;                                  // [2][MAX_N]

  // Role index: hardware warps 4..7 run the single-thread producer / MMA-issue loops, warps 0..3 the epilogue.
  // The SMSP arbiter favours the higher warp id, and each issuer shares its SMSP with one epilogue warp, so this
  // order keeps the ALU-heavy epilogue from starving the issue loops that feed the tensor pipe.
  const int warp = (threadIdx.x >> 5) ^ 4;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.tmA0);
    tma_prefetch_desc(&p.tmW);
    if (p.n_pairs > 1) tma_prefetch_desc(&p.tmA1);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < MAX_STAGES; ++s) {
      mbar_init(bars + s * 8, 2);        // full: A producer + W producer (each arrive.expect_tx)
      mbar_init(bars + 64 + s * 8, MT);  // empty: one tcgen05.commit per MMA issuer
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(bars + 128 + a * 8, MT);           // accumulators full: one commit per issuer
      mbar_init(bars + 144 + a * 8, (EPI_THREADS / 32) * EG);  // accumulators drained (one arrive per epilogue warp)
    }
    mbar_fence_init();
  }
  if (warp == 2) {
    tmem_alloc(smem_u32(tmem_ptr_s), static_cast<uint32_t>(p.tmem_cols));
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_s;
  if (threadIdx.x == 0) TL_MARK(p, TL_SETUP);
  // PDL: everything above (barrier init, TMEM allocation, descriptor prefetch) may overlap the previous kernel of
  // the stream; let the next kernel start its own prologue on idle SMs, then wait for our producer to finish before
  // any activation memory is touched (packed weights / bias are static and need no wait).
  griddep_launch_dependents();
  if (warp != 2) griddep_wait();   // the W producer only reads static data: it runs ahead of the previous kernel's tail
  if (threadIdx.x == 0) TL_MARK(p, TL_DEP);

  // Loop-invariant parameters live in registers: every asm volatile("memory") below would otherwise force the
  // compiler to re-read them from the constant bank inside the issue loops.
  const int num_tiles = p.num_tiles, grid = gridDim.x;
  const int num_n_tiles = p.num_n_tiles, n_tiles_per_group = p.n_tiles_per_group, block_n = p.block_n;
  const int tiles_x = p.tiles_x, tiles_y = p.tiles_y;
  const int n_cblk = p.n_cblk, n_pairs = p.n_pairs, num_stages = p.num_stages, stage_bytes = p.stage_bytes;
  constexpr int KY = MODE == 0 ? 3 : MODE == 1 ? 2 : 1;
  constexpr int KX = KY;
  constexpr uint32_t W_OFF = MT * A_BYTES;
  constexpr int STW = TILE_W * MT;   // super-tile width

  if (warp == 0) {
    // ===================================================== A-tile TMA producer
    int stage = 0;
    uint32_t phase = 0;
    const int pa0 = p.pair_a[0], pa1 = p.pair_a[1], pa2 = p.pair_a[2];
    TileWalker tw_;
    tw_.init(blockIdx.x, grid, num_n_tiles, tiles_x, tiles_y);
    for (int tile = blockIdx.x; tile < num_tiles; tile += grid, tw_.next()) {
      const TileCoord t = tw_.coord_groups(block_n, n_tiles_per_group, STW, TILE_H);
      for (int pair = 0; pair < n_pairs; ++pair) {
        const int pa = pair == 0 ? pa0 : pair == 1 ? pa1 : pa2;
        const CUtensorMap* tmA = pa ? &p.tmA1 : &p.tmA0;
#pragma unroll
        for (int ky = 0; ky < KY; ++ky) {
#pragma unroll
          for (int kx = 0; kx < KX; ++kx) {
            for (int cb = 0; cb < n_cblk; ++cb) {
              mbar_wait(bars + 64 + stage * 8, phase ^ 1u);
              if (elect_one()) {
                const uint32_t full = bars + stage * 8;
                const uint32_t a_dst = smem_base + stage * stage_bytes;
                mbar_arrive_expect_tx(full, MT * A_BYTES);
#pragma unroll
                for (int j = 0; j < MT; ++j) {
                  const int xj = t.x0 + j * TILE_W;
                  if (MODE == 0)
                    tma_load_4d(a_dst + j * A_BYTES, tmA, full, cb * BLOCK_K, xj + kx - 1, t.y0 + ky - 1, t.b);
                  else if (MODE == 1)
                    tma_load_5d(a_dst + j * A_BYTES, tmA, full, cb * BLOCK_K, kx, xj, ky, t.y0);
                  else
                    tma_load_4d(a_dst + j * A_BYTES, tmA, full, cb * BLOCK_K, xj, t.y0, t.b);
                }
              }
              __syncwarp();
              if (++stage == num_stages) {
                stage = 0;
                phase ^= 1u;
              }
            }
          }
        }
      }
    }
  } else if (warp == 2) {
    // ===================================================== W-tile TMA producer
    int stage = 0;
    uint32_t phase = 0;
    const uint32_t w_bytes = static_cast<uint32_t>(block_n * 128);
    const int wg = p.wgroups;
    const int pw0 = p.pair_w[0] * wg, pw1 = p.pair_w[1] * wg, pw2 = p.pair_w[2] * wg;
    TileWalker tw_;
    tw_.init(blockIdx.x, grid, num_n_tiles, tiles_x, tiles_y);
    for (int tile = blockIdx.x; tile < num_tiles; tile += grid, tw_.next()) {
      const TileCoord t = tw_.coord_groups(block_n, n_tiles_per_group, STW, TILE_H);
      for (int pair = 0; pair < n_pairs; ++pair) {
        const int wbase = pair == 0 ? pw0 : pair == 1 ? pw1 : pw2;
#pragma unroll
        for (int tap = 0; tap < KY * KX; ++tap) {
          const int wslice = wbase + (MODE == 2 ? t.grp : tap);
          for (int cb = 0; cb < n_cblk; ++cb) {
            mbar_wait(bars + 64 + stage * 8, phase ^ 1u);
            if (elect_one()) {
              const uint32_t full = bars + stage * 8;
              mbar_arrive_expect_tx(full, w_bytes);
              tma_load_3d(smem_base + stage * stage_bytes + W_OFF, &p.tmW, full, cb * BLOCK_K, t.n0, wslice);
            }
            __syncwarp();
            if (++stage == num_stages) {
              stage = 0;
              phase ^= 1u;
            }
          }
        }
      }
    }
  } else if (warp == 1 || (warp == 3 && MT == 2)) {
    // ===================================================== MMA issuer of sub-tile j (independent accumulators)
    const int j = warp == 1 ? 0 : 1;
    const uint32_t idesc = make_idesc_f16(static_cast<uint32_t>(p.fmt), static_cast<uint32_t>(block_n));
    const int k_iters = n_pairs * p.taps * n_cblk;
    const int last_k16 = p.last_k16;
    const uint32_t a_off = static_cast<uint32_t>(j * A_BYTES);
    int stage = 0;
    uint32_t phase = 0;
    int local_tile = 0;
    uint32_t ready = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += grid, ++local_tile) {
      const int acc = local_tile & 1;
      const uint32_t acc_phase = (local_tile >> 1) & 1;
      mbar_wait(bars + 144 + acc * 8, acc_phase ^ 1u);
      const uint32_t d = tmem_base + static_cast<uint32_t>((acc * MT + j) * block_n);
      uint32_t accumulate = 0;
      int cb = 0;
      for (int kit = 0; kit < k_iters; ++kit) {
        if (!ready) mbar_wait(bars + stage * 8, phase);
        tc_fence_after();
        const uint32_t s_addr = smem_base + stage * stage_bytes;
        const uint32_t empty_bar = bars + 64 + stage * 8;
        const bool full_block = (cb != n_cblk - 1) || (last_k16 == BLOCK_K / 16);
        if (++stage == num_stages) {
          stage = 0;
          phase ^= 1u;
        }
        // peek at the next stage's barrier now; its latency hides behind the MMA issue below
        ready = mbar_test_wait(bars + stage * 8, phase);
        if (elect_one()) {
          const uint64_t adesc = make_sw128_desc(s_addr + a_off, 1024);
          const uint64_t bdesc = make_sw128_desc(s_addr + W_OFF, 1024);
          if (full_block) {
            umma_f16(d, adesc, bdesc, idesc, accumulate);
            umma_f16(d, adesc + 2, bdesc + 2, idesc, 1u);
            umma_f16(d, adesc + 4, bdesc + 4, idesc, 1u);
            umma_f16(d, adesc + 6, bdesc + 6, idesc, 1u);
          } else {
            for (int k = 0; k < last_k16; ++k) umma_f16(d, adesc + 2 * k, bdesc + 2 * k, idesc, k == 0 ? accumulate : 1u);
          }
          umma_commit(empty_bar);                                     // frees the smem stage once these MMAs retire
          if (kit == k_iters - 1) umma_commit(bars + 128 + acc * 8);  // accumulator complete -> epilogue
        }
        __syncwarp();
        accumulate = 1;
        if (++cb == n_cblk) cb = 0;
      }
    }
  } else if (warp >= 4) {
    // ======================================================= epilogue
    const int we = warp & 3;  // TMEM lane quarter this warp may access
    const int eg = (EG == 2 && warp >= 8) ? 1 : 0;   // column half drained by this warp group
    const int row = we * 32 + lane;
    const int th = row / TILE_W, tw = row - th * TILE_W;
    const int et = (threadIdx.x & (EPI_THREADS - 1)) + eg * EPI_THREADS;   // hardware threads 0..127 (+ 256..383)
    const EpiArgs ea = make_epi_args(p);
    const int H = p.H, W = p.W, cout = p.cout;
    const float* bias = p.bias;
    const float* slope = p.slope;
    const bool up = p.wgroups == 4 && MODE == 2;
    const bool staged = p.epi_staged;
    uint8_t* stg = smem_gen + RING_BYTES + (eg * 4 + we) * 4096;
    const int ncols = block_n / EG, col0 = eg * ncols;   // this group's share of the accumulator columns
    const bool one_n_tile = n_tiles_per_group == 1;
    if (one_n_tile) stage_bias_slope(epi_bias, epi_slope, bias, slope, 0, block_n, cout, et, EPI_THREADS * EG);
    int local_tile = 0;
    uint32_t satm = 0;
    TileWalker tw_;
    tw_.init(blockIdx.x, grid, num_n_tiles, tiles_x, tiles_y);
    for (int tile = blockIdx.x; tile < num_tiles; tile += grid, ++local_tile, tw_.next()) {
      const TileCoord t = tw_.coord_groups(block_n, n_tiles_per_group, STW, TILE_H);
      const int acc = local_tile & 1;
      const uint32_t acc_phase = (local_tile >> 1) & 1;
      // bias / slopes depend on the tile's N offset only (not on the transposed conv's phase): staged once when every
      // group has a single N tile — ncu showed the per-tile global loads (long_sb on the staging STS) on the epilogue's
      // critical path of the short-K transposed convs
      float* bs = epi_bias + (one_n_tile ? 0 : acc * MAX_N);
      float* ss = epi_slope + (one_n_tile ? 0 : acc * MAX_N);
      if (!one_n_tile) stage_bias_slope(bs, ss, bias, slope, t.n0, block_n, cout, et, EPI_THREADS * EG);

      mbar_wait(bars + 128 + acc * 8, acc_phase);
      tc_fence_after();

#pragma unroll 1
      for (int j = 0; j < MT; ++j) {
        const int y = t.y0 + th, x = t.x0 + j * TILE_W + tw;
        const bool valid = (y < H) && (x < W);
        const int64_t res_pix = (static_cast<int64_t>(t.b) * H + y) * W + x;
        int64_t out_pix = res_pix;
        if (up) {
          const int ky = t.grp >> 1, kx = t.grp & 1;
          out_pix = (static_cast<int64_t>(t.b) * (2 * H) + (2 * y + ky)) * (2 * W) + (2 * x + kx);
        }
        const uint32_t taddr =
            tmem_base + (static_cast<uint32_t>(we * 32) << 16) + static_cast<uint32_t>((acc * MT + j) * block_n + col0);
        const uint32_t rel = j == MT - 1 ? bars + 144 + acc * 8 : 0u;
        if (MODE == 2 && p.up_fold) {
          // columns = [phase 0 | 1 | 2 | 3] x cout: this group drains phases 2 eg and 2 eg + 1 (EG == 2: MT == 1)
#pragma unroll 1
          for (int q = 0; q < 4 / EG; ++q) {
            const int ph = eg * (4 / EG) + q, ky = ph >> 1, kx = ph & 1;
            const uint32_t tq = taddr + static_cast<uint32_t>(q * cout);
            const uint32_t relq = q == 4 / EG - 1 ? rel : 0u;
            if (staged) {
              RowMap rm;
              rm.b = t.b, rm.y0 = t.y0, rm.x0 = t.x0 + j * TILE_W, rm.tw_shift = 4, rm.H = H, rm.W = W;
              rm.up = 1, rm.ky = ky, rm.kx = kx;
              epilogue_subtile_staged(ea, tq, cout, bs, ss, rm, we * 32, lane, 0, relq, stg, satm);
            } else {
              const int64_t op = (static_cast<int64_t>(t.b) * (2 * H) + (2 * y + ky)) * (2 * W) + (2 * x + kx);
              epilogue_subtile(ea, tq, cout, bs, ss, valid, t.b, y, x, op, res_pix, 0, relq, satm);
            }
          }
        } else if (staged) {
          RowMap rm;
          rm.b = t.b, rm.y0 = t.y0, rm.x0 = t.x0 + j * TILE_W, rm.tw_shift = 4, rm.H = H, rm.W = W;
          rm.up = up ? 1 : 0, rm.ky = t.grp >> 1, rm.kx = t.grp & 1;
          epilogue_subtile_staged(ea, taddr, ncols, bs + col0, ss + col0, rm, we * 32, lane, t.n0 + col0, rel, stg, satm);
        } else {
          epilogue_subtile(ea, taddr, ncols, bs + col0, ss + col0, valid, t.b, y, x, out_pix, res_pix, t.n0 + col0, rel, satm);
        }
      }
    }
    sat_report(ea.sat_flag, satm);
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, static_cast<uint32_t>(p.tmem_cols));
  }
  if (threadIdx.x == 0) TL_MARK(p, TL_EXIT);
}

// ------------------------------------------------------------------ host side
PFN_cuTensorMapEncodeTiled g_encode = nullptr;
std::once_flag g_encode_once;

int get_encoder() {
  std::call_once(g_encode_once, [] {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      g_encode = reinterpret_cast<PFN_cuTensorMapEncodeTiled>(fn);
  });
  if (!g_encode) {
    set_error("cuTensorMapEncodeTiled entry point not available (no CUDA driver?)");
    return B200DN_E_CUDA;
  }
  return 0;
}

int encode(CUtensorMap* tm, CUtensorMapDataType dt, int rank, const void* base, const uint64_t* dims,
           const uint64_t* strides_bytes, const uint32_t* box, const char* what,
           CUtensorMapL2promotion promo = CU_TENSOR_MAP_L2_PROMOTION_L2_256B) {
  uint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = g_encode(tm, dt, static_cast<cuuint32_t>(rank), const_cast<void*>(base), dims, strides_bytes, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, promo,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(%s) failed with CUresult %d (rank %d dims %llu %llu %llu %llu %llu)", what,
              static_cast<int>(r), rank, (unsigned long long)dims[0], (unsigned long long)dims[1],
              (unsigned long long)(rank > 2 ? dims[2] : 0), (unsigned long long)(rank > 3 ? dims[3] : 0),
              (unsigned long long)(rank > 4 ? dims[4] : 0));
    return B200DN_E_CUDA;
  }
  return 0;
}

SmemOptIn g_smem_opt_in;

// default conv3x3 implementation: 1 = per-tap reload (this file), 2 = haloed slab (conv3x3_slab_sm100.cu);
// B200DN_CONV3X3_IMPL=tap|slab overrides, b200dn_igemm_args.impl overrides both.
int default_conv3x3_impl() {
  static int impl = [] {
    const char* e = getenv("B200DN_CONV3X3_IMPL");
    if (e && !strcmp(e, "tap")) return 1;
    if (e && !strcmp(e, "slab")) return 2;
    return B200DN_DEFAULT_CONV3X3_IMPL;
  }();
  return impl;
}
// B200DN_EPI_STAGED: 0 = never, 1 = whenever legal, 2 = only one-accumulator (MT = 1) tiles
int staged_mode() {
  static int mode = [] {
    const char* e = getenv("B200DN_EPI_STAGED");
    return e ? atoi(e) : 2;
  }();
  return mode;
}
bool wres_enabled() {
  static int on = [] {
    const char* e = getenv("B200DN_SLAB_WRES");
    return e ? atoi(e) : 1;
  }();
  return on != 0;
}
// B200DN_CTA2: 0 = never use the CTA-pair slab kernel, 1 = whenever legal (default), 2 = only when every SM pair gets a tile
int cta2_mode() {
  static int mode = [] {
    const char* e = getenv("B200DN_CTA2");
    return e ? atoi(e) : 1;
  }();
  return mode;
}
// B200DN_UP_FOLD=0: transposed convs keep one tile per output phase even when all four fit one accumulator
int up_fold_enabled() {
  static int v = [] {
    const char* e = getenv("B200DN_UP_FOLD");
    return e ? atoi(e) : 1;
  }();
  return v;
}
// B200DN_SPLIT_N: smallest N tile the under-filled-grid heuristic may choose (default 64; 0 or 256 = never split)
int split_n_floor() {
  static int v = [] {
    const char* e = getenv("B200DN_SPLIT_N");
    const int x = e ? atoi(e) : 64;
    return x <= 0 ? 256 : x < 16 ? 16 : x;
  }();
  return v;
}
// B200DN_W_ROW_STAGES: 1 (default) = a streamed-W ring stage holds a filter row (3 taps) when N <= 64
bool w_row_stages() {
  static int on = [] {
    const char* e = getenv("B200DN_W_ROW_STAGES");
    return e ? atoi(e) : 1;
  }();
  return on != 0;
}
// B200DN_SLAB_PITCH: slab row pitch in pixels, 10 (default) .. 16 (the first version's layout)
int slab_pitch() {
  static int w = [] {
    const char* e = getenv("B200DN_SLAB_PITCH");
    const int v = e ? atoi(e) : 10;
    return v < 10 ? 10 : v > 16 ? 16 : v;
  }();
  return w;
}
// B200DN_L2PROMO: L2 promotion of the activation tensor maps, 0 none / 1 64 B / 2 128 B / 3 256 B
CUtensorMapL2promotion a_l2_promotion() {
  static int v = [] {
    const char* e = getenv("B200DN_L2PROMO");
    return e ? atoi(e) : 3;
  }();
  return v == 0 ? CU_TENSOR_MAP_L2_PROMOTION_NONE : v == 1 ? CU_TENSOR_MAP_L2_PROMOTION_L2_64B
       : v == 2 ? CU_TENSOR_MAP_L2_PROMOTION_L2_128B : CU_TENSOR_MAP_L2_PROMOTION_L2_256B;
}

}  // namespace

// Validate `a`, choose the kernel family / tiling / ring sizes and — unless this is a plan-only query (`info` set) —
// encode the tensor maps and resolve the kernel variant into `cfg`.
int igemm_configure(const b200dn_igemm_args& a, LaunchCfg* cfg, b200dn_igemm_plan_info* info, int sms_override) {
  B200DN_CHECK_ARG(a.mode >= 0 && a.mode <= 3, "igemm: bad mode %d", a.mode);
  B200DN_CHECK_ARG(a.prec >= 0 && a.prec <= 4, "igemm: bad prec %d", a.prec);
  B200DN_CHECK_ARG(a.B > 0 && a.H > 0 && a.W > 0 && a.cin > 0 && a.cout > 0, "igemm: non-positive dims");
  B200DN_CHECK_ARG(a.in[0] && a.wpacked && a.bias, "igemm: null input/weight/bias pointer");
  B200DN_CHECK_ARG(a.in_ctot % 8 == 0 && a.in_ctot >= a.cin, "igemm: in_ctot %d must be a multiple of 8 and >= cin %d",
                   a.in_ctot, a.cin);
  B200DN_CHECK_ARG(a.impl >= 0 && a.impl <= 3, "igemm: bad impl %d", a.impl);
  const bool two_a = (a.prec == B200DN_PREC_BF16X2 || a.prec == B200DN_PREC_BF16X3 || a.prec == B200DN_PREC_FP16X2);
  const bool two_w = (a.prec == B200DN_PREC_BF16X3);
  B200DN_CHECK_ARG(!two_a || a.in[1], "igemm: prec %d needs the lo activation plane in[1]", a.prec);
  if (a.mode == B200DN_MODE_DOWN2X2)
    B200DN_CHECK_ARG(a.H % 2 == 0 && a.W % 2 == 0, "igemm: DOWN2X2 needs even H, W (got %d x %d)", a.H, a.W);
  if (info == nullptr) {   // plan-only calls never touch the device
    B200DN_CHECK_ARG(cfg != nullptr, "igemm: internal: no launch configuration to fill");
    if (int rc = require_sm100()) return rc;
    if (int rc = get_encoder()) return rc;
  } else {
    B200DN_CHECK_ARG(sms_override > 0, "igemm_plan: sm_count must be positive");
  }
  const int impl = a.impl ? a.impl : default_conv3x3_impl();
  const bool slab = a.mode == B200DN_MODE_CONV3X3 && impl >= 2;

  KParams p_local;
  KParams& p = cfg ? cfg->p : p_local;
  memset(&p, 0, sizeof(p));
  p.sat_flag = a.sat_flag;
  p.taps = a.mode == B200DN_MODE_CONV3X3 ? 9 : a.mode == B200DN_MODE_DOWN2X2 ? 4 : 1;
  p.wgroups = a.mode == B200DN_MODE_CONV3X3 ? 9 : a.mode == B200DN_MODE_CONV1X1 ? 1 : 4;
  const int n_groups = a.mode == B200DN_MODE_UP2X2 ? 4 : 1;
  if (a.mode == B200DN_MODE_DOWN2X2) {
    p.B = 1;
    p.H = a.B * (a.H / 2);
    p.W = a.W / 2;
  } else {
    p.B = a.B;
    p.H = a.H;
    p.W = a.W;
  }
  p.n_cblk = cdiv(a.cin, BLOCK_K);
  p.last_k16 = cdiv(a.cin - (p.n_cblk - 1) * BLOCK_K, 16);
  p.cout = a.cout;
  const int cin_pad = round_up(a.cin, BLOCK_K);
  const int cout_pad = round_up(a.cout, 16);
  int sms = info ? sms_override : device_sm_count();
  if (sms <= 0) return B200DN_E_CUDA;
  int block_n = a.block_n;
  // Transposed conv whose four phases fit one accumulator (4 * cout <= 256, cout a multiple of 16: level 1 -> 0 of
  // base_filters <= 32): N = [phase 0 | 1 | 2 | 3] in one tile.  The A tile is loaded once instead of four times and
  // the per-tile pipeline round trips (4 UMMAs of K = 64 each) are paid once per pixel tile.
  const bool up_fold = a.mode == B200DN_MODE_UP2X2 && block_n == 0 && a.m_tiles != 2 && up_fold_enabled() &&
                       a.cout % 16 == 0 && 4 * a.cout <= MAX_N;
  if (up_fold) block_n = 4 * a.cout;
  if (block_n == 0) {
    const int nt = cdiv(cout_pad, MAX_N);
    block_n = round_up(cdiv(cout_pad, nt), 16);
    // Under-filled grid (batch 1-2, the deep levels): split N further, down to 64, until every SM has a tile (B200DN_SPLIT_N).  The
    // reference's own scripts run batch_size = 1 (evaluate_model.py:318, evaluate_SIDD.py:116); there a level-3 layer
    // has 8 pixel tiles, and 8 x (1024 / 256) tiles would leave 116 of 148 SMs idle.
    const int th0 = a.mode == B200DN_MODE_CONV3X3 ? SLAB_TILE_H : TILE_H, tw0 = a.mode == B200DN_MODE_CONV3X3 ? SLAB_TILE_W : TILE_W;
    const int64_t m_tiles1 = static_cast<int64_t>(p.B) * cdiv(p.W, tw0) * cdiv(p.H, th0);
    const int groups = a.mode == B200DN_MODE_UP2X2 ? 4 : 1;
    while (block_n >= split_n_floor() * 2 && (block_n / 2) % 16 == 0 && cout_pad % (block_n / 2) == 0 &&
           m_tiles1 * cdiv(cout_pad, block_n) * groups < sms)
      block_n /= 2;
  }
  B200DN_CHECK_ARG(block_n % 16 == 0 && block_n >= 16 && block_n <= MAX_N, "igemm: block_n %d invalid", block_n);
  p.block_n = block_n;
  p.up_fold = up_fold ? 1 : 0;
  p.n_tiles_per_group = up_fold ? 1 : cdiv(cout_pad, block_n);
  p.num_n_tiles = up_fold ? 1 : p.n_tiles_per_group * n_groups;
  // accumulator tile: 16 x 8 pixels (tap kernel, sub-tiles side by side) or 8 x 16 (slab kernel, sub-tiles stacked)
  const int tw1 = slab ? SLAB_TILE_W : TILE_W, th1 = slab ? SLAB_TILE_H : TILE_H;
  // two A tiles per W tile (M = 256) when N is small enough for 4 accumulators in TMEM and there is enough
  // work to keep every SM busy with the halved tile count
  int mt = a.m_tiles;
  B200DN_CHECK_ARG(mt >= 0 && mt <= 2, "igemm: m_tiles %d invalid", mt);
  if (mt == 2) B200DN_CHECK_ARG(block_n <= 128, "igemm: m_tiles=2 needs block_n <= 128 (TMEM columns)");
  if (mt == 0) {
    const int64_t tiles2 = slab ? static_cast<int64_t>(p.B) * cdiv(p.W, tw1) * cdiv(p.H, 2 * th1) * p.num_n_tiles
                                : static_cast<int64_t>(p.B) * cdiv(p.W, 2 * tw1) * cdiv(p.H, th1) * p.num_n_tiles;
    mt = (block_n <= 128 && tiles2 >= 2 * sms) ? 2 : 1;
    // transposed conv (short K = Cin, epilogue-bound): one accumulator per W tile, drained by two epilogue groups,
    // measured 7-15 % faster than MT = 2 at every width (profiles/r02_up_conv_variants.txt)
    if (a.mode == B200DN_MODE_UP2X2) mt = 1;
  }
  p.mt = mt;
  const int stw = slab ? tw1 : tw1 * mt, sth = slab ? th1 * mt : th1;   // super-tile extent
  p.tiles_x = cdiv(p.W, stw);
  p.tiles_y = cdiv(p.H, sth);
  p.num_m_tiles = p.B * p.tiles_x * p.tiles_y;
  p.num_tiles = p.num_m_tiles * p.num_n_tiles;
  p.fmt = (a.prec == B200DN_PREC_FP16 || a.prec == B200DN_PREC_FP16X2) ? 0 : 1;
  switch (a.prec) {
    case B200DN_PREC_BF16X2:
    case B200DN_PREC_FP16X2:
      p.n_pairs = 2;
      p.pair_w[0] = 0, p.pair_a[0] = 1;  // small term first
      p.pair_w[1] = 0, p.pair_a[1] = 0;
      break;
    case B200DN_PREC_BF16X3:
      p.n_pairs = 3;
      p.pair_w[0] = 1, p.pair_a[0] = 0;
      p.pair_w[1] = 0, p.pair_a[1] = 1;
      p.pair_w[2] = 0, p.pair_a[2] = 0;
      break;
    default:
      p.n_pairs = 1;
      p.pair_w[0] = 0, p.pair_a[0] = 0;
  }
  if (slab) {
    // Slab row pitch in pixels (SBO = pitch * 128 B).  The 8-wide tile needs 10 (one halo pixel each side); the swizzle
    // XOR of TMA and UMMA follows absolute shared-memory address bits, so the pitch need not be a multiple of the
    // 8-row swizzle atom.  10 instead of 16 cuts the slab's L2->SM bytes and shared-memory writes by 37.5 % and makes
    // room for a deeper ring (more loads in flight per SM; the F = 32 level-0 layers were waiting on slab data).
    p.slab_w = slab_pitch();
    p.slab_tx = p.slab_w * (SLAB_TILE_H * mt + 2) * 128;
    p.slab_bytes = round_up(p.slab_tx, 1024);
    p.n_wplanes = two_w ? 2 : 1;
    const int64_t w_all = static_cast<int64_t>(p.n_wplanes) * p.n_cblk * 9 * block_n * 128;
    // small layers: keep the whole packed weight set resident in shared memory (single N tile only; cout < 64: such
    // layers never use the staged epilogue, so its 16 KB belong to the resident weights) next to >= 2 slabs
    // N = 32..48 layers with K >= 9 * 64 on a full grid go to the CTA-pair kernel instead (measured 7-14 % faster than
    // resident weights at cin 64..128 / 256x256 and 128x128, slower at cin 32; profiles/r02_n32_pairs_vs_wres.txt)
    const int pair_tiles0 = cdiv(p.num_m_tiles, 2) * p.num_n_tiles;
    const bool small_n_pairs = a.impl == 0 && cta2_mode() >= 1 && block_n >= 32 && block_n < 64 && a.cin >= 64 &&
                               pair_tiles0 >= sms / 2;
    p.wres = (impl != 3 && !small_n_pairs && p.num_n_tiles == 1 && block_n < 64 &&
              w_all <= SLAB_WRES_BYTES - 2 * p.slab_bytes && wres_enabled()) ? 1 : 0;
    // CTA pairs (cta_group::2, conv3x3_slab2_kernel): each SM keeps half of every W tile.  Explicit impl 3, or by
    // default for the streaming-weight layers (N >= 64): when every SM pair gets at least one pair tile, and also
    // when the grid is under-filled anyway (batch 1-2, deep levels) — there each CTA is paced by the latency of its
    // own weight stream, which a pair halves, and 2 x pair tiles keep as many SMs busy as single-CTA tiles would.
    const int pair_tiles = cdiv(p.num_m_tiles, 2) * p.num_n_tiles;
    const bool pairs_fit = pair_tiles >= sms / 2 || (cta2_mode() == 1 && p.num_tiles < sms && p.num_m_tiles >= 2);
    p.cta2 = (!p.wres && block_n >= 32 &&
              (impl == 3 || small_n_pairs || (a.impl == 0 && cta2_mode() >= 1 && block_n >= 64 && pairs_fit))) ? 1 : 0;
    if (p.cta2) p.num_tiles = pair_tiles;
    p.w_taps = 1;
    if (p.wres) {
      p.num_slabs = static_cast<int>((SLAB_WRES_BYTES - w_all) / p.slab_bytes);
      p.stage_bytes = block_n * 128;
      p.num_stages = 1;
    } else {
      // W ring: one tap tile per stage, or a whole filter row (3 taps) per stage for N <= 64, where the per-stage
      // barrier traffic of the issuer warp costs as much as the UMMAs it guards.  4 stages (N = 256) .. 8 stages;
      // the slabs take the rest.
      p.w_taps = (block_n <= 64 && w_row_stages()) ? 3 : 1;
      p.stage_bytes = (p.cta2 ? block_n / 2 : block_n) * 128 * p.w_taps;
      int want = p.w_taps == 3 ? (p.cta2 ? 5 : 4) : block_n > 128 ? 4 : block_n > 64 ? 6 : 8;
      p.num_slabs = (SLAB_DATA_BYTES - want * p.stage_bytes) / p.slab_bytes;
      if (p.num_slabs < 2) p.num_slabs = 2;
      if (p.num_slabs > SLAB_MAX_SLABS) p.num_slabs = SLAB_MAX_SLABS;
      p.num_stages = (SLAB_DATA_BYTES - p.num_slabs * p.slab_bytes) / p.stage_bytes;
      if (p.num_stages > MAX_STAGES) p.num_stages = MAX_STAGES;
    }
    if (p.num_slabs > SLAB_MAX_SLABS) p.num_slabs = SLAB_MAX_SLABS;
  } else {
    p.stage_bytes = mt * A_BYTES + block_n * 128;
    p.num_stages = RING_BYTES / p.stage_bytes;
    if (p.num_stages > MAX_STAGES) p.num_stages = MAX_STAGES;
  }
  int cols = 32;
  while (cols < 2 * mt * block_n) cols <<= 1;
  p.tmem_cols = cols;

  p.bias = a.bias;
  p.slope = a.slope;
  p.out_kind = a.out_kind;
  // staged (smem-transposed, 128-byte-row) epilogue: single-plane NHWC output in whole 64-channel groups
  // (the one-accumulator transposed-conv variant splits the columns over two epilogue groups: 64-channel groups per half)
  const int epi_cols = up_fold ? a.cout : (a.mode == B200DN_MODE_UP2X2 && mt == 1) ? block_n / 2 : block_n;
  p.epi_staged = (a.out_kind == B200DN_OUT_NHWC16 && !two_a && epi_cols % 64 == 0 && a.cout % 64 == 0 &&
                  a.out_coff % 64 == 0 && a.out_ctot % 8 == 0 && (staged_mode() == 1 || (staged_mode() == 2 && mt == 1))) ? 1 : 0;
  if (a.out_kind == B200DN_OUT_NHWC16) {
    B200DN_CHECK_ARG(a.out[0], "igemm: null NHWC output");
    B200DN_CHECK_ARG(!two_a || a.out[1], "igemm: prec %d needs the lo output plane out[1]", a.prec);
    B200DN_CHECK_ARG(a.out_ctot % 8 == 0 && a.out_coff % 8 == 0 && a.cout % 8 == 0 &&
                         a.out_coff + a.cout <= a.out_ctot,
                     "igemm: NHWC output slice [%d,%d) of %d must be 8-channel aligned", a.out_coff,
                     a.out_coff + a.cout, a.out_ctot);
    p.out0 = a.out[0];
    p.out1 = two_a ? a.out[1] : nullptr;
    p.out_ctot = a.out_ctot;
    p.out_coff = a.out_coff;
    if (a.res[0]) {
      B200DN_CHECK_ARG(a.mode == B200DN_MODE_CONV3X3 || a.mode == B200DN_MODE_CONV1X1,
                       "igemm: NHWC residual only with stride-1 modes");
      B200DN_CHECK_ARG(a.res_ctot % 8 == 0 && a.res_ctot >= a.cout, "igemm: bad res_ctot %d", a.res_ctot);
      B200DN_CHECK_ARG(!two_a || a.res[1], "igemm: prec %d needs the lo residual plane", a.prec);
      p.res0 = a.res[0];
      p.res1 = two_a ? a.res[1] : nullptr;
      p.res_ctot = a.res_ctot;
    }
  } else if (a.out_kind == B200DN_OUT_NCHW32) {
    B200DN_CHECK_ARG(a.out_nchw, "igemm: null NCHW output");
    B200DN_CHECK_ARG(a.mode == B200DN_MODE_CONV3X3 || a.mode == B200DN_MODE_CONV1X1,
                     "igemm: NCHW output only with stride-1 modes");
    p.out_nchw = a.out_nchw;
    p.res_nchw = a.res_nchw;
    p.res_bmod = a.res_bmod > 0 ? a.res_bmod : a.B;
  } else {
    B200DN_CHECK_ARG(false, "igemm: bad out_kind %d", a.out_kind);
  }

  int grid = p.num_tiles < sms ? p.num_tiles : sms;
  if (a.max_ctas > 0 && grid > a.max_ctas) grid = a.max_ctas;
  int clusters = 0;
  if (slab && p.cta2) {
    clusters = p.num_tiles < sms / 2 ? p.num_tiles : sms / 2;
    if (a.max_ctas > 0 && clusters > (a.max_ctas + 1) / 2) clusters = (a.max_ctas + 1) / 2;
  }
  if (info != nullptr) {
    memset(info, 0, sizeof(*info));
    info->kernel = slab ? (p.cta2 ? 2 : 1) : 0;
    info->mt = mt, info->block_n = block_n, info->num_n_tiles = p.num_n_tiles, info->num_tiles = p.num_tiles;
    info->grid = (slab && p.cta2) ? 2 * clusters : grid;
    info->wres = p.wres, info->num_slabs = slab ? p.num_slabs : 0, info->slab_bytes = slab ? p.slab_bytes : 0;
    info->num_stages = p.num_stages, info->stage_bytes = p.stage_bytes, info->w_taps = slab ? p.w_taps : 1;
    info->tmem_cols = p.tmem_cols, info->epi_staged = p.epi_staged;
    if (slab) {
      const int w_bytes = p.wres ? p.n_wplanes * p.n_cblk * 9 * block_n * 128 : p.num_stages * p.stage_bytes;
      info->data_bytes_used = p.num_slabs * p.slab_bytes + w_bytes;
      info->data_bytes_budget = p.wres ? SLAB_WRES_BYTES : SLAB_DATA_BYTES;
    } else {
      info->data_bytes_used = p.num_stages * p.stage_bytes;
      info->data_bytes_budget = RING_BYTES;
    }
    return 0;
  }

  // ---- tensor maps
  const CUtensorMapDataType dt = p.fmt ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  const uint64_t ct = static_cast<uint64_t>(a.in_ctot);
  for (int pl = 0; pl < (two_a ? 2 : 1); ++pl) {
    CUtensorMap* tm = pl ? &p.tmA1 : &p.tmA0;
    B200DN_CHECK_ARG((reinterpret_cast<uintptr_t>(a.in[pl]) & 15) == 0, "igemm: input plane %d not 16-byte aligned", pl);
    if (a.mode == B200DN_MODE_DOWN2X2) {
      // (c, kx, ox, ky, b*Ho+oy): address = ((2*oy'+ky)*W + 2*ox+kx)*ctot + c
      uint64_t dims[5] = {static_cast<uint64_t>(a.cin), 2, static_cast<uint64_t>(a.W / 2), 2,
                          static_cast<uint64_t>(a.B) * (a.H / 2)};
      uint64_t str[4] = {ct * 2, 2 * ct * 2, static_cast<uint64_t>(a.W) * ct * 2, 2 * static_cast<uint64_t>(a.W) * ct * 2};
      uint32_t box[5] = {BLOCK_K, 1, TILE_W, 1, TILE_H};
      if (int rc = encode(tm, dt, 5, a.in[pl], dims, str, box, "A/down", a_l2_promotion())) return rc;
    } else {
      uint64_t dims[4] = {static_cast<uint64_t>(a.cin), static_cast<uint64_t>(a.W), static_cast<uint64_t>(a.H),
                          static_cast<uint64_t>(a.B)};
      uint64_t str[3] = {ct * 2, static_cast<uint64_t>(a.W) * ct * 2,
                         static_cast<uint64_t>(a.H) * static_cast<uint64_t>(a.W) * ct * 2};
      uint32_t box[4] = {BLOCK_K, TILE_W, TILE_H, 1};
      if (slab) {
        box[1] = static_cast<uint32_t>(p.slab_w);
        box[2] = static_cast<uint32_t>(SLAB_TILE_H * mt + 2);
      }
      if (int rc = encode(tm, dt, 4, a.in[pl], dims, str, box, slab ? "A/slab" : "A", a_l2_promotion())) return rc;
    }
  }
  {
    B200DN_CHECK_ARG((reinterpret_cast<uintptr_t>(a.wpacked) & 15) == 0, "igemm: packed weights not 16-byte aligned");
    uint64_t dims[3] = {static_cast<uint64_t>(cin_pad), static_cast<uint64_t>(cout_pad),
                        static_cast<uint64_t>(p.wgroups) * (two_w ? 2 : 1)};
    uint64_t str[2] = {static_cast<uint64_t>(cin_pad) * 2, static_cast<uint64_t>(cin_pad) * cout_pad * 2};
    // resident mode: all 9 taps per box; streamed: w_taps taps per box; CTA pairs: half of the N rows per CTA
    uint32_t box[3] = {BLOCK_K, static_cast<uint32_t>(p.cta2 ? block_n / 2 : block_n),
                       p.wres ? 9u : static_cast<uint32_t>(slab ? p.w_taps : 1)};
    if (up_fold) box[1] = static_cast<uint32_t>(a.cout), box[2] = 4;   // [phase][cout] rows = the N = 4 * cout tile
    if (int rc = encode(&p.tmW, dt, 3, a.wpacked, dims, str, box, "W")) return rc;
  }

  cfg->kind = 0;
  cfg->cooperative = 0;
#ifdef B200DN_TIMELINE
  {
    char label[96];
    snprintf(label, sizeof(label), "%s %dx%dx%d cin %d cout %d N %d mt %d %s", a.mode == B200DN_MODE_CONV3X3 ? "conv3x3"
             : a.mode == B200DN_MODE_DOWN2X2 ? "down" : "up", a.B, a.H, a.W, a.cin, a.cout, block_n, mt,
             slab ? (p.cta2 ? "pairs" : p.wres ? "wres" : "slab") : "tap");
    p.tl = igemm::timeline_slots(label);
  }
#endif
  if (slab && p.cta2) return resolve_conv3x3_slab2(cfg, 2 * clusters);
  if (slab) return resolve_conv3x3_slab(cfg, grid);

  static const void* const kernels[6] = {
      reinterpret_cast<const void*>(igemm_kernel<0, 1>), reinterpret_cast<const void*>(igemm_kernel<0, 2>),
      reinterpret_cast<const void*>(igemm_kernel<1, 1>), reinterpret_cast<const void*>(igemm_kernel<1, 2>),
      reinterpret_cast<const void*>(igemm_kernel<2, 1>), reinterpret_cast<const void*>(igemm_kernel<2, 2>)};
  if (int rc = ensure_max_dyn_smem(g_smem_opt_in, kernels, 6, SMEM_BYTES, "cudaFuncSetAttribute(igemm_kernel, smem)"))
    return rc;
  const int mode_idx = a.mode == B200DN_MODE_CONV3X3 ? 0 : a.mode == B200DN_MODE_DOWN2X2 ? 1 : 2;
  cfg->kernel = kernels[mode_idx * 2 + (mt - 1)];
  cfg->grid = grid;
  cfg->threads = NUM_THREADS + ((mode_idx == 2 && mt == 1) ? EPI_THREADS : 0);
  cfg->smem = SMEM_BYTES;
  cfg->cluster = 1;
  return 0;
}

int igemm_launch_cfg(const LaunchCfg& cfg, cudaStream_t stream) {
  // the parameter block is copied by the launch itself; nothing is re-encoded here
  void* params = cfg.kind == 1   ? static_cast<void*>(const_cast<FusedParams*>(&cfg.f))
                 : cfg.kind == 2 ? static_cast<void*>(const_cast<ChainParams*>(&cfg.c))
                                 : static_cast<void*>(const_cast<KParams*>(&cfg.p));
  B200DN_CUDA(launch_pdl(cfg.kernel, cfg.grid, cfg.threads, static_cast<size_t>(cfg.smem), stream, params, cfg.cluster,
                         cfg.cooperative != 0));
  return 0;
}

namespace igemm {
#ifdef B200DN_TIMELINE
namespace {
constexpr int TL_MAX_LAUNCHES = 4096;
unsigned long long* g_tl_base = nullptr;
std::vector<std::string> g_tl_labels;
std::mutex g_tl_mutex;
}  // namespace
unsigned long long* timeline_slots(const char* label) {
  std::lock_guard<std::mutex> lock(g_tl_mutex);
  if (g_tl_base == nullptr) {
    if (cudaMalloc(&g_tl_base, TL_MAX_LAUNCHES * 16 * sizeof(unsigned long long)) != cudaSuccess) return nullptr;
    cudaMemset(g_tl_base, 0, TL_MAX_LAUNCHES * 16 * sizeof(unsigned long long));
  }
  if (static_cast<int>(g_tl_labels.size()) >= TL_MAX_LAUNCHES) return nullptr;
  g_tl_labels.emplace_back(label);
  return g_tl_base + (g_tl_labels.size() - 1) * 16;
}
#endif
int get_tensor_map_encoder(PFN_encodeTiled* fn) {
  if (int rc = get_encoder()) return rc;
  *fn = g_encode;
  return 0;
}
}  // namespace igemm

}  // namespace b200dn

#ifdef B200DN_TIMELINE
// diagnostics build only (not in include/b200dn.h): one line per configured launch, the 9 slots in ns relative to `t0`
extern "C" int b200dn_debug_timeline_dump(const char* path) {
  using namespace b200dn::igemm;
  std::lock_guard<std::mutex> lock(g_tl_mutex);
  if (g_tl_base == nullptr) return -1;
  cudaDeviceSynchronize();
  const size_t n = g_tl_labels.size();
  std::vector<unsigned long long> h(n * 16);
  if (cudaMemcpy(h.data(), g_tl_base, n * 16 * sizeof(unsigned long long), cudaMemcpyDeviceToHost) != cudaSuccess) return -2;
  FILE* f = fopen(path, "w");
  if (!f) return -3;
  fprintf(f, "# launch entry setup dep mma0 mma_end acc0 epi_end exit sm | label   (ns, absolute %%globaltimer; 0 = not recorded)\n");
  for (size_t i = 0; i < n; ++i) {
    fprintf(f, "%zu", i);
    for (int k = 0; k < 9; ++k) fprintf(f, " %llu", h[i * 16 + k]);
    fprintf(f, " | %s\n", g_tl_labels[i].c_str());
  }
  fclose(f);
  return static_cast<int>(n);
}
#endif

// the opaque handle of include/b200dn.h
struct b200dn_igemm_prepared {
  b200dn::igemm::LaunchCfg cfg;
  int out_kind;
};

extern "C" int b200dn_igemm_plan(const b200dn_igemm_args* args, int sm_count, b200dn_igemm_plan_info* info) {
  if (!args || !info) {
    b200dn::set_error("igemm_plan: null args / info");
    return B200DN_E_ARG;
  }
  return b200dn::igemm_configure(*args, nullptr, info, sm_count);
}

extern "C" int b200dn_igemm(const b200dn_igemm_args* args, void* stream) {
  if (!args) {
    b200dn::set_error("igemm: null args");
    return B200DN_E_ARG;
  }
  b200dn::igemm::LaunchCfg cfg;
  if (int rc = b200dn::igemm_configure(*args, &cfg)) return rc;
  return b200dn::igemm_launch_cfg(cfg, static_cast<cudaStream_t>(stream));
}

extern "C" int b200dn_igemm_prepare(const b200dn_igemm_args* args, b200dn_igemm_prepared** out) {
  if (!args || !out) {
    b200dn::set_error("igemm_prepare: null args / out");
    return B200DN_E_ARG;
  }
  *out = nullptr;
  b200dn_igemm_prepared* h = new (std::nothrow) b200dn_igemm_prepared();     // value-initialised: no field of the launch configuration is left indeterminate
  if (!h) {
    b200dn::set_error("igemm_prepare: out of host memory");
    return B200DN_E_ARG;
  }
  if (int rc = b200dn::igemm_configure(*args, &h->cfg)) {
    delete h;
    return rc;
  }
  h->out_kind = args->out_kind;
  *out = h;
  return 0;
}

extern "C" int b200dn_dense_block_prepare(const b200dn_dense_block_args* args, b200dn_igemm_prepared** out) {
  if (!args || !out) {
    b200dn::set_error("dense_block_prepare: null args / out");
    return B200DN_E_ARG;
  }
  *out = nullptr;
  b200dn::igemm::PFN_encodeTiled enc = nullptr;
  if (args->channels == 32 && (args->prec == B200DN_PREC_BF16 || args->prec == B200DN_PREC_FP16) && args->in && args->out) {
    if (int rc = b200dn::require_sm100()) return rc;
    if (int rc = b200dn::igemm::get_tensor_map_encoder(&enc)) return rc;
  }
  b200dn_igemm_prepared* h = new (std::nothrow) b200dn_igemm_prepared();     // value-initialised: no field of the launch configuration is left indeterminate
  if (!h) {
    b200dn::set_error("dense_block_prepare: out of host memory");
    return B200DN_E_ARG;
  }
  if (int rc = b200dn::igemm::configure_dense_block(*args, &h->cfg, enc)) {
    delete h;
    return rc;
  }
  h->out_kind = B200DN_OUT_NHWC16;
  *out = h;
  return 0;
}

extern "C" int b200dn_dense_block_set_epilogue_constants(b200dn_igemm_prepared* prep, const float* const* bias_host,
                                                         const float* const* slope_host) {
  if (!prep || prep->cfg.kind != 1 || !prep->cfg.alt_kernel) {
    b200dn::set_error("dense_block_set_epilogue_constants: not a prepared dense block");
    return B200DN_E_ARG;
  }
  if (!bias_host || !slope_host) {
    b200dn::set_error("dense_block_set_epilogue_constants: null argument");
    return B200DN_E_ARG;
  }
  for (int j = 0; j < 4; ++j)
    if (!bias_host[j] || !slope_host[j]) {
      b200dn::set_error("dense_block_set_epilogue_constants: null bias / slope %d", j);
      return B200DN_E_ARG;
    }
  b200dn::igemm::FusedParams& f = prep->cfg.f;
  // accumulator-column order [o0 (16) | o1 (16) | o2 (16) | o3 (32)]
  for (int c = 0; c < 80; ++c) {
    const int j = c < 48 ? c >> 4 : 3, k = c < 48 ? c & 15 : c - 48;
    f.cbias[c] = bias_host[j][k];
    f.cslope[c] = slope_host[j][k];
  }
  if (!f.epi_const) {
    f.epi_const = 1;
    prep->cfg.kernel = prep->cfg.alt_kernel;
  }
  return 0;
}

extern "C" int64_t b200dn_conv_chain_workspace_bytes(const b200dn_igemm_args* layers, int n_layers) {
  if (!layers || n_layers < 1) {
    b200dn::set_error("conv_chain_workspace_bytes: bad arguments");
    return B200DN_E_ARG;
  }
  return static_cast<int64_t>(b200dn::igemm::conv_chain_workspace_bytes(layers, n_layers));
}

extern "C" int b200dn_conv_chain_prepare(const b200dn_igemm_args* layers, int n_layers, void* workspace, int flags,
                                         b200dn_igemm_prepared** out) {
  if (!layers || !out) {
    b200dn::set_error("conv_chain_prepare: null layers / out");
    return B200DN_E_ARG;
  }
  *out = nullptr;
  b200dn_igemm_prepared* h = new (std::nothrow) b200dn_igemm_prepared();     // value-initialised: no field of the launch configuration is left indeterminate
  if (!h) {
    b200dn::set_error("conv_chain_prepare: out of host memory");
    return B200DN_E_ARG;
  }
  if (int rc = b200dn::igemm::configure_conv_chain(layers, n_layers, workspace, flags, &h->cfg)) {
    delete h;
    return rc;
  }
  h->out_kind = B200DN_OUT_NHWC16;
  *out = h;
  return 0;
}

extern "C" int b200dn_igemm_rebind_nchw(b200dn_igemm_prepared* prep, float* out_nchw, const float* res_nchw, int res_bmod) {
  if (!prep || prep->out_kind != B200DN_OUT_NCHW32 || !out_nchw) {
    b200dn::set_error("igemm_rebind_nchw: needs a prepared OUT_NCHW32 launch and a non-null output");
    return B200DN_E_ARG;
  }
  prep->cfg.p.out_nchw = out_nchw;
  prep->cfg.p.res_nchw = res_nchw;
  if (res_bmod > 0) prep->cfg.p.res_bmod = res_bmod;
  return 0;
}

extern "C" int b200dn_igemm_launch(const b200dn_igemm_prepared* prep, void* stream) {
  if (!prep) {
    b200dn::set_error("igemm_launch: null handle");
    return B200DN_E_ARG;
  }
  return b200dn::igemm_launch_cfg(prep->cfg, static_cast<cudaStream_t>(stream));
}

extern "C" int b200dn_igemm_launch_list(b200dn_igemm_prepared* const* preps, int n, void* stream) {
  if (!preps || n < 0) {
    b200dn::set_error("igemm_launch_list: bad arguments");
    return B200DN_E_ARG;
  }
  for (int i = 0; i < n; ++i) {
    if (!preps[i]) {
      b200dn::set_error("igemm_launch_list: null handle at %d", i);
      return B200DN_E_ARG;
    }
    if (int rc = b200dn::igemm_launch_cfg(preps[i]->cfg, static_cast<cudaStream_t>(stream))) return rc;
  }
  return 0;
}

extern "C" void b200dn_igemm_release(b200dn_igemm_prepared* prep) { delete prep; }

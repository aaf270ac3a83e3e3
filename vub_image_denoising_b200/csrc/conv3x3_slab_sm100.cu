// conv3x3_slab_sm100.cu — 3x3 / stride 1 / pad 1 convolution as a tcgen05 implicit GEMM that loads every input
// pixel into shared memory ONCE per 64-channel block instead of once per filter tap.  One kernel body, three launches:
//   conv3x3_slab_kernel<MT, WRES>   one CTA per tile; resident weights (WRES) for the small layers; the output block
//   conv3x3_slab2_kernel<MT>        CTA pairs (`cta_group::2`, M = 256 per instruction, cluster of 2)
//   conv3x3_chain_kernel<MT>        2..4 dependent layers of one resolution in one persistent launch, on CTA pairs
//
// Reference op: nn.Conv2d(.,.,3,padding=1) + nn.PReLU (+ dense-block residual / output-block residual),
// UNet/RDUNet_model.py:61,74-75,86-87,98-115,186 — 63 of the network's 69 convolutions, 97.5 % of its FLOPs.
//
// Why: the per-tap kernel (igemm_sm100.cu) is bound by shared-memory bandwidth — every pipeline stage writes
// an A tile (TMA) that is read by only four UMMAs, and TMA writes + UMMA operand reads share ~128 B/clk/SM.
// Here one TMA box brings a haloed slab [ (16*MT+2) rows x slab_w px x 64 ch ] (zero-filled outside the image = the
// conv's padding); the 9 taps are 9 UMMA descriptors into that slab, shifted by (dy*slab_w + dx) rows of 128 B.
// The slab pitch slab_w is 10 pixels (the 8-pixel tile + halo; B200DN_SLAB_PITCH selects up to 16), so the 8-row
// core-matrix groups of a tap sit slab_w * 128 B apart (SBO).  Measured on B200 (tools/slab_probe.py): the 128B-swizzle
// XOR of both TMA and UMMA is a function of the ABSOLUTE shared memory address bits [7,10), so a descriptor whose start
// address is shifted by whole 128 B rows reads the TMA-written slab correctly with the descriptor's base-offset field
// left at 0 (setting it to (addr >> 7) & 7 produces garbage).
// A-side smem write traffic drops 4x, A TMA instructions 9x, L2->SM traffic ~4x.
//
// Warp roles: 0 = slab TMA producer, 2 = TMEM allocator then W-tile TMA producer (one [N x 64] tile per tap),
// 1 / 3 = MMA issuers of sub-tile 0 / 1 (MT = 2 stacks two 8x16-pixel tiles vertically), 4..7 = epilogue.
//
// CTA pairs.  With cta_group::1 every UMMA re-reads its whole B operand ([N x 16] weights) from the issuing SM's shared
// memory, and the N = 64 / 128 layers are bound by shared-memory bandwidth (A 4 KB + B N*32 B per UMMA against
// ~128 B/clk/SM; DESIGN.md §3.1).  In a CTA pair each SM keeps only HALF of the W tile (rows [r*N/2, (r+1)*N/2)) and
// the hardware shares the halves across the pair, so per SM the W smem reads, the W TMA writes and the L2->SM weight
// traffic all halve, while each CTA still owns its pixels (slab), its accumulators (TMEM) and its epilogue.
// Protocol (rank 0 = leader):
//   * both CTAs run the slab producer and the W producer into their OWN shared memory, but every TMA credits its bytes
//     to the LEADER's full barrier (`.cta_group::2` TMA + mapa address);
//   * only the leader's issuer warps issue MMAs; `tcgen05.commit ... multicast::cluster` with mask 0b11 arrives on the
//     empty / accumulator-full barriers at the same offset in BOTH CTAs;
//   * both epilogues drain their own TMEM and release the accumulator stage by a remote arrive on the leader's barrier
//     (one relaxed arrive per epilogue warp, count = 2 x 4).
// Tile schedule: pair tile = (two consecutive spatial super tiles, one N tile); clusters take pair tiles round-robin.
//
// Chains.  Launched one by one every layer pays, on top of its MMAs, a drain (the last tile's epilogue, 1.5-12 us),
// the hand-off to the dependent launch (1-3 us after the last CTA exits) and a cold pipeline fill (first TMA
// 1-2.5 us): ~7 us per layer at 32 images (10 % of the RDUNet_T(32) forward), ~4 us of every ~10 us layer at 2 images
// (profiles/r02_launch_timeline_*.txt).  A chain makes the layers of a DenoisingBlock (conv_0..conv_3, every conv
// reading the block input plus all earlier outputs = channel slices of one NHWC buffer) ONE work list, layer-major:
// item = (layer, pair tile), cluster c takes items c, c + G, c + 2G, ...; a tile of layer k only needs the 3 x 3
// neighbourhood of spatial tiles of layer k - 1 (its 1-pixel halo), so it waits on per-tile arrival counters in global
// memory instead of a grid-wide boundary.  The TMA / MMA / epilogue pipelines of a CTA never drain between layers, the
// weights of the next layer stream in while the current one computes, and tiles of layer k + 1 start while other
// SMs still finish layer k.  Per item, on top of the CTA-pair protocol:
//   * slab producer, layer k > 0: nine lanes poll the counters of layer k - 1 for the tile's 3 x 3 neighbourhood
//     (ld.acquire.gpu) until each holds epoch x (N tiles x 4 epilogue warps) arrivals, then fence.proxy.async and the
//     TMA.  By induction the neighbourhood is then complete for every earlier layer too.
//   * epilogue warp, layer k < last: after its stores, __threadfence + one red.add on its tile's counter.
//   * counters are monotonic; `epoch` (launches completed + 1) is read from the workspace at kernel start and advanced
//     by the last CTA to leave, so nothing is reset between launches and a graph replay needs no memset node.
// Deadlock freedom: a cluster runs its items in increasing order and an item only waits on lower-numbered items, so the
// lowest unfinished item can always run — provided every cluster becomes resident: the grid is clamped to
// cudaOccupancyMaxActiveClusters, and clusters that find their SMs taken by the previous launch of the stream start
// when it drains (it never waits on this one).  What this does NOT cover is a second chain launch on ANOTHER stream
// of the same device holding SMs while it waits for its own clusters: chain launches of one device must not overlap
// (one plan = one stream here).  B200DN_CHAIN_COOP=1 launches cooperatively (all-or-nothing residency), which lifts
// that restriction but cannot be profiled: ncu 2025.2 fails cooperative cluster launches with LaunchFailed.
// Polls are bounded by the same watchdog as the mbarrier waits (trap, not hang).
// The chain runs the same kernel body, tiles and MMA order as the per-layer launches: outputs are bit-equal.
#include "igemm_common.cuh"

#include <type_traits>

namespace b200dn {
namespace igemm {

namespace {

constexpr int TW = SLAB_TILE_W;   // 8
constexpr int TH = SLAB_TILE_H;   // 16
constexpr int MAX_SLABS = SLAB_MAX_SLABS;
constexpr int DATA_BYTES = SLAB_DATA_BYTES + EPI_STAGING_BYTES;   // [slabs | W ring or resident W | epilogue staging]
// after the barriers: bias / PReLU slopes, [2][MAX_N] each (per N tile, double-buffered), or [CHAIN_MAX_LAYERS][MAX_N]
// (a chain stages every layer once)
constexpr int slab_smem_bytes(int bias_slots) { return 1024 + DATA_BYTES + SLAB_CTRL_BYTES + 2 * bias_slots * MAX_N * 4; }
constexpr int SMEM_BYTES_SLAB = slab_smem_bytes(2);
constexpr int SMEM_BYTES_CHAIN = slab_smem_bytes(CHAIN_MAX_LAYERS);

// barrier map (byte offsets from `bars`): up to 8 slab slots and 8 W stages
constexpr uint32_t B_SLAB_FULL = 0, B_SLAB_EMPTY = 64, B_W_FULL = 128, B_W_EMPTY = 192, B_TFULL = 256, B_TEMPTY = 272,
                   B_TMEM_PTR = 288;

// WRES: the layer's whole packed weight set ([w plane][64-ch block][tap][N x 64]) is loaded into shared memory once
// per CTA and stays resident; the main loop then only streams slabs.  Used for the small layers (F = 32 levels 0/1),
// which are latency-bound: per tile it removes 9 W-tile round trips and keeps the issue loop small enough for the
// instruction cache (ncu: the unrolled 9-tap path showed mostly `no_inst` stalls there).
// Epilogue warp groups: the resident-weight layers (N <= 48, K <= 9 * 128) do so little tensor work per output that
// the epilogue's CUDA-core instruction stream is what paces a tile (measured: time proportional to pixels, independent
// of K, of MT and of DRAM vs L2 residency; 4 epilogue warps run at ~0.27 IPC each).  With MT = 2 a second group of four
// warps (hardware warps 8..11) drains sub-tile 1 while the first drains sub-tile 0.
template <int MT, bool WRES>
constexpr int slab_epi_groups() { return (WRES && MT == 2) ? 2 : 1; }

// ---- work lists ------------------------------------------------------------------------------------------------
// A role loop runs over items first, first + stride, ... < num_items and asks its walker for each item's layer and
// tile.  The one-layer walkers are division-free and their layer is the constant 0; a chain decodes every item.
struct Work {
  int layer;
  bool live;     // the tile lies in the batch (not the odd CTA of the last pair)
  TileCoord t;   // live == false: an all-out-of-bounds tile (TMA zero-fills, the epilogue masks every pixel)
  int b, ty, tx, m;   // chain: spatial tile digits, for the dependency counters
};

// one CTA per tile: TileWalker (igemm_common.cuh)
struct SoloWalker {
  TileWalker w;
  __device__ __forceinline__ void init(const KParams& p, int first, int stride, int) {
    w.init(first, stride, p.num_n_tiles, p.tiles_x, p.tiles_y);
  }
  __device__ __forceinline__ void next() { w.next(); }
  __device__ __forceinline__ Work at(const KParams& p, int, int tile_h) const {
    Work k;
    k.layer = 0, k.live = true, k.t = w.coord(p.block_n, TW, tile_h);
    return k;
  }
};

// CTA pairs: the walk over the pair tiles cluster_id, cluster_id + num_clusters, ... : pair tile = (m_pair, N tile),
// this CTA's spatial super tile is m_tile = 2 * m_pair + rank (an all-out-of-bounds tile past the end for the odd CTA
// of the last pair).  The strides are decomposed once into (tile column, tile row, image) digits and added with carries.
struct PairWalker {
  int nt, tx, ty, b;
  int s_nt, d_tx, d_ty, d_b, e_tx, e_ty, e_b;   // stride digits: N tile; 2 * pair stride; the extra 2 on an N-tile carry
  int num_n_tiles, tiles_x, tiles_y, images;
  __device__ __forceinline__ static void split(int m, int tiles_x, int tiles_y, int& tx, int& ty, int& b) {
    const int q = m / tiles_x;
    tx = m - q * tiles_x;
    b = q / tiles_y;
    ty = q - b * tiles_y;
  }
  __device__ __forceinline__ void init(const KParams& p, int pair_tile, int stride, int rank) {
    num_n_tiles = p.num_n_tiles, tiles_x = p.tiles_x, tiles_y = p.tiles_y, images = p.B;
    const int m_pair = pair_tile / num_n_tiles;
    nt = pair_tile - m_pair * num_n_tiles;
    split(2 * m_pair + rank, tiles_x, tiles_y, tx, ty, b);
    const int s_pair = stride / num_n_tiles;
    s_nt = stride - s_pair * num_n_tiles;
    split(2 * s_pair, tiles_x, tiles_y, d_tx, d_ty, d_b);
    split(2, tiles_x, tiles_y, e_tx, e_ty, e_b);
  }
  __device__ __forceinline__ void add(int ax, int ay, int ab) {
    tx += ax;
    int c = tx >= tiles_x ? 1 : 0;
    tx -= c ? tiles_x : 0;
    ty += ay + c;
    c = ty >= tiles_y ? 1 : 0;
    ty -= c ? tiles_y : 0;
    b += ab + c;
  }
  __device__ __forceinline__ void next() {
    nt += s_nt;
    const bool carry = nt >= num_n_tiles;
    nt -= carry ? num_n_tiles : 0;
    add(d_tx, d_ty, d_b);
    if (carry) add(e_tx, e_ty, e_b);
  }
  __device__ __forceinline__ Work at(const KParams& p, int, int tile_h) const {
    Work k;
    k.layer = 0, k.live = true;
    k.t.grp = 0, k.t.n0 = nt * p.block_n;
    if (b >= images) {
      k.t.b = 0, k.t.x0 = 0, k.t.y0 = tiles_y * tile_h;
    } else {
      k.t.b = b, k.t.y0 = ty * tile_h, k.t.x0 = tx * TW;
    }
    return k;
  }
};

__device__ __forceinline__ int chain_layer(const ChainParams& c, int item) {
  return (item >= c.item_base[1] ? 1 : 0) + (item >= c.item_base[2] ? 1 : 0) + (item >= c.item_base[3] ? 1 : 0);
}

// chain: item -> (layer, N tile, this CTA's spatial super tile of the pair tile)
struct ChainWalker {
  int rank;
  __device__ __forceinline__ void init(const ChainParams&, int, int, int rank_) { rank = rank_; }
  __device__ __forceinline__ void next() {}
  __device__ __forceinline__ Work at(const ChainParams& c, int item, int tile_h) const {
    Work k;
    k.layer = chain_layer(c, item);
    const KParams& p = c.L[k.layer];
    const int pt = item - c.item_base[k.layer];
    const int m_pair = pt / p.num_n_tiles;
    k.t.grp = 0, k.t.n0 = (pt - m_pair * p.num_n_tiles) * p.block_n;
    k.m = 2 * m_pair + rank;
    const int q = k.m / p.tiles_x;
    k.tx = k.m - q * p.tiles_x;
    k.b = q / p.tiles_y;
    k.ty = q - k.b * p.tiles_y;
    k.live = k.b < c.L[0].B;
    k.t.y0 = k.live ? k.ty * tile_h : p.tiles_y * tile_h, k.t.x0 = k.live ? k.tx * TW : 0, k.t.b = k.live ? k.b : 0;
    return k;
  }
};

// parameters of the layer of a work item, and those that hold for the whole launch
__device__ __forceinline__ const KParams& layer_params(const KParams& p, int) { return p; }
__device__ __forceinline__ const KParams& layer_params(const ChainParams& c, int layer) { return c.L[layer]; }
__device__ __forceinline__ int num_items(const KParams& p) { return p.num_tiles; }
__device__ __forceinline__ int num_items(const ChainParams& c) { return c.item_base[c.n_layers]; }
__device__ __forceinline__ int acc_columns(const KParams& p) { return p.block_n; }
__device__ __forceinline__ int acc_columns(const ChainParams& c) { return c.nmax; }   // the chain's largest N
__device__ __forceinline__ void prefetch_tensor_maps(const KParams& p) {
  tma_prefetch_desc(&p.tmA0);
  tma_prefetch_desc(&p.tmW);
  if (p.n_pairs > 1) tma_prefetch_desc(&p.tmA1);
}
__device__ __forceinline__ void prefetch_tensor_maps(const ChainParams& c) {
  for (int l = 0; l < c.n_layers; ++l) {
    tma_prefetch_desc(&c.L[l].tmA0);
    tma_prefetch_desc(&c.L[l].tmW);
  }
}

// ---- CTA group: one CTA per MMA, or a pair ------------------------------------------------------------------------
// Arm `full` for `tx` bytes and load one TMA box into this CTA's shared memory.  CTA pair: both CTAs' boxes credit the
// LEADER's barrier, which the leader alone arms for the bytes of both.
// (3 coordinates: a W box, 4: a slab box)
template <int CTAS, class... C>
__device__ __forceinline__ void tma_box(uint32_t dst, const CUtensorMap* tm, uint32_t full, uint32_t tx, bool leader,
                                        C... c) {
  if (CTAS == 1 || leader) mbar_arrive_expect_tx(full, tx);
  if constexpr (CTAS == 2 && sizeof...(C) == 3) tma_load_3d_2sm(dst, tm, mapa_shared(full, 0), c...);
  if constexpr (CTAS == 2 && sizeof...(C) == 4) tma_load_4d_2sm(dst, tm, mapa_shared(full, 0), c...);
  if constexpr (CTAS == 1 && sizeof...(C) == 3) tma_load_3d(dst, tm, full, c...);
  if constexpr (CTAS == 1 && sizeof...(C) == 4) tma_load_4d(dst, tm, full, c...);
}
// CTA pair: arrives on the barrier at the same offset in both CTAs
template <int CTAS>
__device__ __forceinline__ void mma_commit(uint32_t bar) {
  if constexpr (CTAS == 2)
    umma_commit_2cta(bar, 3);
  else
    umma_commit(bar);
}
// CTA pair: the barrier inits and the TMEM allocation of BOTH CTAs are visible before any remote arrive; at exit,
// neither CTA may leave (or free its TMEM) while the other can still read its shared memory through an MMA or signal
// one of its barriers
template <int CTAS>
__device__ __forceinline__ void group_sync() {
  if constexpr (CTAS == 2)
    cluster_sync_all();
  else
    __syncthreads();
}

// per-layer constants of the MMA issuer
struct IssueShape {
  uint32_t idesc;
  int n_cblk, kc_iters, last_k16, w_taps;
  uint64_t tap_step;   // descriptor units between the tap tiles of a W stage (this CTA's half of a tile on a pair)
};
template <int CTAS, bool CHAIN>
__device__ __forceinline__ IssueShape issue_shape(const KParams& p) {
  IssueShape s;
  s.idesc = make_idesc_f16(static_cast<uint32_t>(p.fmt), static_cast<uint32_t>(p.block_n), BLOCK_M * CTAS);
  s.n_cblk = p.n_cblk;
  s.kc_iters = CHAIN ? p.n_cblk : p.n_pairs * p.n_cblk;   // a chain's layers have one plane pair
  s.last_k16 = p.last_k16;
  s.w_taps = p.w_taps;
  if constexpr (CTAS == 1)
    s.tap_step = static_cast<uint64_t>(static_cast<uint32_t>(p.block_n * 128) >> 4);
  else
    s.tap_step = static_cast<uint64_t>(((p.block_n >> 1) * 128) >> 4);
  return s;
}

// ---- chain dependencies -----------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t ld_acquire_gpu(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void red_add_gpu(uint32_t* p, uint32_t v) {
  asm volatile("red.relaxed.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

// Wait until layer `layer`'s outputs exist on the 3 x 3 spatial tiles around (b, ty, tx): lanes 0..8 poll one counter each.
__device__ __forceinline__ void wait_neighbourhood(const ChainParams& c, int layer, const Work& it, uint32_t epoch, int lane) {
  const KParams& p = c.L[layer];
  if (lane < 9) {
    const int dy = lane / 3 - 1, dx = lane - (lane / 3) * 3 - 1;
    const int ny = it.ty + dy, nx = it.tx + dx;
    if (ny >= 0 && ny < p.tiles_y && nx >= 0 && nx < p.tiles_x) {
      const uint32_t* f = c.flags + static_cast<size_t>(layer) * p.num_m_tiles + ((it.b * p.tiles_y + ny) * p.tiles_x + nx);
      const uint32_t need = epoch * static_cast<uint32_t>(c.flag_need[layer]);
      if (static_cast<int32_t>(ld_acquire_gpu(f) - need) < 0) {
        const long long t0 = clock64();
        uint32_t spins = 0;
        while (static_cast<int32_t>(ld_acquire_gpu(f) - need) < 0) {
          if ((++spins & 0xff) == 0 && (clock64() - t0) > B200DN_WATCHDOG_CYCLES) {
            printf("b200dn: conv chain watchdog (block %d layer %d tile %d,%d,%d)\n", (int)blockIdx.x, layer, it.b, ny, nx);
            __trap();
          }
        }
      }
    }
  }
  __syncwarp();
  asm volatile("fence.proxy.async;" ::: "memory");   // generic-proxy writes of other SMs -> this SM's TMA reads
}

// ---- the kernel body ----------------------------------------------------------------------------------------------
// MT: 128-pixel sub-tiles per W tile; CTAS: CTAs per MMA (2 = cta_group::2); WRES: resident weights (one CTA, one
// layer); P: KParams (one layer) or ChainParams (a chain).  Every difference between the variants is resolved at
// compile time: the issue loop in particular must stay on the uniform datapath (DESIGN.md §3.2).
template <int MT, int CTAS, bool WRES, class P>
__device__ __forceinline__ void conv3x3_slab_body(const P& prm) {
  constexpr bool CHAIN = std::is_same_v<P, ChainParams>;
  static_assert(!WRES || (CTAS == 1 && !CHAIN), "resident weights: one CTA, one layer");
  static_assert(!CHAIN || CTAS == 2, "chains run on CTA pairs");
  constexpr int EG = slab_epi_groups<MT, WRES>();
  constexpr int STH = TH * MT;
  using Walker = std::conditional_t<CHAIN, ChainWalker, std::conditional_t<CTAS == 2, PairWalker, SoloWalker>>;
  const KParams& p0 = layer_params(prm, 0);   // a chain's ring geometry is common to its layers (the host unified it)

  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_u32 = smem_u32(smem_raw);
  const uint32_t smem_base = (raw_u32 + 1023u) & ~1023u;
  if (threadIdx.x == 0) TL_MARK(p0, TL_ENTRY);
  uint8_t* smem_gen = smem_raw + (smem_base - raw_u32);
  const uint32_t bars = smem_base + DATA_BYTES;
  uint32_t* tmem_ptr_s = reinterpret_cast<uint32_t*>(smem_gen + DATA_BYTES + B_TMEM_PTR);
  float* epi_bias = reinterpret_cast<float*>(smem_gen + DATA_BYTES + SLAB_CTRL_BYTES);
  float* epi_slope = epi_bias + (CHAIN ? CHAIN_MAX_LAYERS : 2) * MAX_N;

  // Role index: hardware warps 4..7 run the single-thread producer / MMA-issue loops, warps 0..3 the epilogue.
  // The SMSP arbiter favours the higher warp id, and each issuer shares its SMSP with one epilogue warp, so this
  // order keeps the ALU-heavy epilogue from starving the issue loops that feed the tensor pipe.
  const int warp = (threadIdx.x >> 5) ^ 4;
  const int lane = threadIdx.x & 31;
  const int rank = CTAS == 2 ? static_cast<int>(cluster_ctarank()) : 0;
  const bool leader = rank == 0;
  const int first = CTAS == 2 ? blockIdx.x >> 1 : blockIdx.x;   // cluster id on a pair
  const int stride = CTAS == 2 ? gridDim.x >> 1 : gridDim.x;

  if (warp == 0 && lane == 0) prefetch_tensor_maps(prm);
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < MAX_SLABS; ++s) {
      mbar_init(bars + B_SLAB_FULL + s * 8, 1);      // on a pair the leader's counts one arrive.expect_tx for both CTAs
      mbar_init(bars + B_SLAB_EMPTY + s * 8, MT);    // one commit per issuer
    }
    for (int s = 0; s < MAX_STAGES; ++s) {
      mbar_init(bars + B_W_FULL + s * 8, 1);
      mbar_init(bars + B_W_EMPTY + s * 8, MT);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(bars + B_TFULL + a * 8, MT);
      mbar_init(bars + B_TEMPTY + a * 8, (EPI_THREADS / 32) * EG * CTAS);   // one arrive per epilogue warp (of both CTAs)
    }
    mbar_fence_init();
  }
  if (warp == 2) {
    if constexpr (CTAS == 2) {
      tmem_alloc_2cta(smem_u32(tmem_ptr_s), static_cast<uint32_t>(prm.tmem_cols));
      tmem_relinquish_2cta();
    } else {
      tmem_alloc(smem_u32(tmem_ptr_s), static_cast<uint32_t>(prm.tmem_cols));
      tmem_relinquish();
    }
  }
  tc_fence_before();
  group_sync<CTAS>();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_s;
  if (threadIdx.x == 0) TL_MARK(p0, TL_SETUP);
  // PDL: everything above (barrier init, TMEM allocation, descriptor prefetch) may overlap the previous kernel of
  // the stream; let the next kernel start its own prologue on idle SMs, then wait for our producer to finish before
  // any activation memory is touched.  The W producer (resident or streamed) only reads the packed weights (static
  // data): it fills its ring while the previous kernel is still running.
  griddep_launch_dependents();
  if (warp != 2) griddep_wait();
  if (threadIdx.x == 0) TL_MARK(p0, TL_DEP);
  [[maybe_unused]] bool tl_first = false;

  const int n_items = num_items(prm);
  const int num_slabs = p0.num_slabs, slab_bytes = p0.slab_bytes;
  const int num_stages = p0.num_stages, stage_bytes = p0.stage_bytes;
  const uint32_t wring = smem_base + static_cast<uint32_t>(num_slabs * slab_bytes);
  const uint32_t acc_stride = static_cast<uint32_t>(acc_columns(prm));   // TMEM columns between accumulators

  if (warp == 0) {
    // ===================================================== slab TMA producer: one box per (plane pair, 64-channel block)
    [[maybe_unused]] uint32_t epoch = 0;
    if constexpr (CHAIN) epoch = *reinterpret_cast<const volatile uint32_t*>(prm.sync) + 1u;
    int s = 0;
    uint32_t sph = 0;
    const int pa0 = p0.pair_a[0], pa1 = p0.pair_a[1], pa2 = p0.pair_a[2];
    Walker wk;
    wk.init(prm, first, stride, rank);
    for (int item = first; item < n_items; item += stride, wk.next()) {
      const Work w = wk.at(prm, item, STH);
      const KParams& p = layer_params(prm, w.layer);
      if constexpr (CHAIN) {
        if (w.layer > 0 && w.live) wait_neighbourhood(prm, w.layer - 1, w, epoch, lane);
      }
      const int n_pairs = CHAIN ? 1 : p.n_pairs, n_cblk = p.n_cblk;
      for (int pair = 0; pair < n_pairs; ++pair) {
        const int pa = pair == 0 ? pa0 : pair == 1 ? pa1 : pa2;
        const CUtensorMap* tmA = (!CHAIN && pa) ? &p.tmA1 : &p.tmA0;
        for (int cb = 0; cb < n_cblk; ++cb) {
          mbar_wait(bars + B_SLAB_EMPTY + s * 8, sph ^ 1u);
          if (elect_one())
            tma_box<CTAS>(smem_base + s * slab_bytes, tmA, bars + B_SLAB_FULL + s * 8,
                          static_cast<uint32_t>(CTAS * p.slab_tx), leader, cb * BLOCK_K, w.t.x0 - 1, w.t.y0 - 1, w.t.b);
          __syncwarp();
          if (++s == num_slabs) {
            s = 0;
            sph ^= 1u;
          }
        }
      }
    }
  } else if (warp == 2) {
    if constexpr (WRES) {
      // ===================================================== resident weights: 9 taps per box, loaded once
      const KParams& p = p0;
      if (elect_one()) {
        const int n_cblk = p.n_cblk, n_boxes = p.n_wplanes * n_cblk;
        const uint32_t box_bytes = static_cast<uint32_t>(9 * p.block_n * 128);
        const uint32_t full = bars + B_W_FULL;
        mbar_arrive_expect_tx(full, static_cast<uint32_t>(n_boxes) * box_bytes);
        for (int wp = 0; wp < p.n_wplanes; ++wp)
          for (int cb = 0; cb < n_cblk; ++cb)
            tma_load_3d(wring + static_cast<uint32_t>(wp * n_cblk + cb) * box_bytes, &p.tmW, full, cb * BLOCK_K, 0,
                        wp * 9);
      }
      __syncwarp();
      griddep_wait();
    } else {
      // ===================================================== W-tile TMA producer: w_taps tap tiles per ring stage
      // (on a pair: this CTA's half of each [N x 64] tile)
      int ws = 0;
      uint32_t wph = 0;
      const int pw0 = p0.pair_w[0] * 9, pw1 = p0.pair_w[1] * 9, pw2 = p0.pair_w[2] * 9;
      Walker wk;
      wk.init(prm, first, stride, rank);
      for (int item = first; item < n_items; item += stride, wk.next()) {
        const Work w = wk.at(prm, item, STH);
        const KParams& p = layer_params(prm, w.layer);
        const int n_pairs = CHAIN ? 1 : p.n_pairs, n_cblk = p.n_cblk, w_taps = p.w_taps;
        const uint32_t w_bytes = static_cast<uint32_t>(p.block_n * 128 * w_taps);   // both halves on a pair
        const int n_row = w.t.n0 + rank * (p.block_n >> 1);
        for (int pair = 0; pair < n_pairs; ++pair) {
          const int wbase = CHAIN ? 0 : pair == 0 ? pw0 : pair == 1 ? pw1 : pw2;
          for (int cb = 0; cb < n_cblk; ++cb) {
#pragma unroll 1
            for (int tap = 0; tap < 9; tap += w_taps) {
              mbar_wait(bars + B_W_EMPTY + ws * 8, wph ^ 1u);
              if (elect_one())
                tma_box<CTAS>(wring + ws * stage_bytes, &p.tmW, bars + B_W_FULL + ws * 8, w_bytes, leader,
                              cb * BLOCK_K, n_row, wbase + tap);
              __syncwarp();
              if (++ws == num_stages) {
                ws = 0;
                wph ^= 1u;
              }
            }
          }
        }
      }
    }
  } else if (leader && (warp == 1 || (warp == 3 && MT == 2))) {
    // ===================================================== MMA issuer of sub-tile j (on a pair: the leader's, for both SMs)
    // The loop is deliberately small: dy rolled, descriptors and barrier addresses advanced incrementally, the k16
    // count of a tap a compile-time constant per code path, and outside a chain only a tile count.  ncu
    // (profiles/r01_n64_issuer_warp_issue_bound_ncu.txt) showed this warp issue-bound — ~130 SASS instructions per tap,
    // never waiting for data — which capped every layer with N <= 64.
    const int j = warp == 1 ? 0 : 1;
    const uint32_t pitch = static_cast<uint32_t>(p0.slab_w * 128);   // bytes per slab pixel row = SBO
    const uint64_t row_step = static_cast<uint64_t>(pitch >> 4);     // descriptor address units (16 B)
    IssueShape sh = issue_shape<CTAS, CHAIN>(p0);
    const int pw_0 = p0.pair_w[0], pw_1 = p0.pair_w[1], pw_2 = p0.pair_w[2];   // resident weights: w plane of a pair
    const uint32_t w_tile_bytes = static_cast<uint32_t>(p0.block_n * 128);
    // streamed-W ring cursor (unused when the weights are resident)
    WRing wr;
    wr.full0 = bars + B_W_FULL, wr.empty0 = bars + B_W_EMPTY;
    wr.full_end = wr.full0 + static_cast<uint32_t>(num_stages) * 8;
    wr.desc0 = make_sw128_desc(wring, 1024);
    wr.step = static_cast<uint64_t>(stage_bytes >> 4);
    wr.full = wr.full0, wr.empty = wr.empty0, wr.phase = 0, wr.desc = wr.desc0;
    if constexpr (WRES) mbar_wait(bars + B_W_FULL, 0);   // resident weights have landed
    int s = 0;
    uint32_t sph = 0;
    int local_tile = 0;
    for (int item = first; item < n_items; item += stride, ++local_tile) {
      if constexpr (CHAIN) sh = issue_shape<CTAS, CHAIN>(prm.L[chain_layer(prm, item)]);
      const int acc = local_tile & 1;
      const uint32_t acc_phase = (local_tile >> 1) & 1;
      mbar_wait(bars + B_TEMPTY + acc * 8, acc_phase ^ 1u);
      tc_fence_after();
      const uint32_t d = tmem_base + static_cast<uint32_t>(acc * MT + j) * acc_stride;
      uint32_t accumulate = 0;
      int cb = 0;
      for (int kc = 0; kc < sh.kc_iters; ++kc) {
        const int nk = (cb != sh.n_cblk - 1) ? BLOCK_K / 16 : sh.last_k16;
        mbar_wait(bars + B_SLAB_FULL + s * 8, sph);
        if (j == 0 && lane == 0) TL_MARK_ONCE(p0, TL_MMA0, tl_first);
        // one CTA: fence here; the pair issuers fence only after each W-stage wait inside the streamed block
        if constexpr (CTAS == 1) tc_fence_after();
        const uint32_t slab = smem_base + static_cast<uint32_t>(s * slab_bytes) + static_cast<uint32_t>(j * TH) * pitch;
        uint64_t arow = make_sw128_desc(slab, pitch);
        if constexpr (WRES) {
          // resident weights: [w plane][cb][tap][N x 64]; pair index = kc / n_cblk
          const int pair = kc / sh.n_cblk;
          const int wpl = pair == 0 ? pw_0 : pair == 1 ? pw_1 : pw_2;
          const uint64_t bdesc = make_sw128_desc(wring + static_cast<uint32_t>((wpl * sh.n_cblk + cb) * 9) * w_tile_bytes, 1024);
          if (elect_one()) {
            switch (nk) {   // one dispatch per 9 taps; inside, the k16 count is a compile-time constant
              case 4: issue_slab_block_resident<4>(d, arow, row_step, bdesc, sh.tap_step, sh.idesc, accumulate); break;
              case 3: issue_slab_block_resident<3>(d, arow, row_step, bdesc, sh.tap_step, sh.idesc, accumulate); break;
              case 2: issue_slab_block_resident<2>(d, arow, row_step, bdesc, sh.tap_step, sh.idesc, accumulate); break;
              default: issue_slab_block_resident<1>(d, arow, row_step, bdesc, sh.tap_step, sh.idesc, accumulate); break;
            }
            umma_commit(bars + B_SLAB_EMPTY + s * 8);
            if (kc == sh.kc_iters - 1) umma_commit(bars + B_TFULL + acc * 8);
          }
          __syncwarp();
          accumulate = 1;
        } else {
          issue_slab_block_streamed_n<CTAS == 2>(nk, sh.w_taps, d, arow, row_step, wr, sh.tap_step, sh.idesc, accumulate);
          if (elect_one()) {
            mma_commit<CTAS>(bars + B_SLAB_EMPTY + s * 8);                         // slab consumed by all 9 taps
            if (kc == sh.kc_iters - 1) mma_commit<CTAS>(bars + B_TFULL + acc * 8);  // accumulator complete
          }
          __syncwarp();
        }
        if (++s == num_slabs) {
          s = 0;
          sph ^= 1u;
        }
        if (++cb == sh.n_cblk) cb = 0;
      }
    }
    if (j == 0 && lane == 0) TL_MARK(p0, TL_MMA_END);
  } else if (warp >= 4) {
    // ======================================================= epilogue (on a pair: each CTA its own accumulators)
    const int we = warp & 3;
    const int row = we * 32 + lane;
    const int th = row / TW, tw = row - th * TW;
    const int eg = (EG == 2 && warp >= 8) ? 1 : 0;    // epilogue group (hardware warps 0..3 / 8..11)
    const int et = (threadIdx.x & (EPI_THREADS - 1)) + eg * EPI_THREADS;
    uint8_t* stg = smem_gen + SLAB_DATA_BYTES + we * 4096;
    const uint32_t tempty = CTAS == 2 ? mapa_shared(bars + B_TEMPTY, 0) : bars + B_TEMPTY;   // the leader's on a pair
    const EpiArgs ea0 = make_epi_args(p0);
    int* sat_flag = ea0.sat_flag;   // a chain reports to the flag of its last item's layer
    // the fp32 NCHW output block (cout <= 4), single-CTA only
    const bool nchw_small = CTAS == 1 && p0.out_kind == B200DN_OUT_NCHW32 && p0.cout <= 4 && p0.block_n == 16;
    const int res_bmod = p0.res_bmod > 0 ? p0.res_bmod : 1;
    const int64_t hw = static_cast<int64_t>(p0.H) * p0.W;
    // bias / PReLU slopes: staged once when the layer has a single N tile, or for a chain once for every layer (static
    // data: the global loads overlap the first accumulator's MMAs); else per tile, double-buffered.  Per-tile global
    // loads + a named barrier are a large share of a tile of the small-K layers.
    const bool one_n_tile = p0.num_n_tiles == 1;
    if constexpr (CHAIN) {
      for (int l = 0; l < prm.n_layers; ++l) {
        const KParams& pl = prm.L[l];
        for (int i = et; i < MAX_N; i += EPI_THREADS) {
          epi_bias[l * MAX_N + i] = i < pl.cout ? __ldg(pl.bias + i) : 0.f;
          epi_slope[l * MAX_N + i] = (pl.slope != nullptr && i < pl.cout) ? __ldg(pl.slope + i) : 1.f;
        }
      }
      asm volatile("bar.sync 1, %0;" ::"r"(EPI_THREADS) : "memory");
    } else if (one_n_tile) {
      stage_bias_slope(epi_bias, epi_slope, p0.bias, p0.slope, 0, p0.block_n, p0.cout, et, EPI_THREADS * EG);
    }
    int local_tile = 0;
    uint32_t satm = 0;
    Walker wk;
    wk.init(prm, first, stride, rank);
    for (int item = first; item < n_items; item += stride, ++local_tile, wk.next()) {
      const Work w = wk.at(prm, item, STH);
      const TileCoord t = w.t;
      const int acc = local_tile & 1;
      const uint32_t acc_phase = (local_tile >> 1) & 1;
      // per-layer values: loop invariants outside a chain
      const KParams& p = layer_params(prm, w.layer);
      const EpiArgs ea = CHAIN ? make_epi_args(p) : ea0;
      const int block_n = p.block_n;
      const bool staged = !WRES && p.epi_staged;
      const float* bs;
      const float* ss;
      if constexpr (CHAIN) {
        sat_flag = ea.sat_flag;
        bs = epi_bias + w.layer * MAX_N + t.n0;
        ss = epi_slope + w.layer * MAX_N + t.n0;
      } else {
        float* bt = epi_bias + (one_n_tile ? 0 : acc * MAX_N);
        float* st = epi_slope + (one_n_tile ? 0 : acc * MAX_N);
        if (!one_n_tile) stage_bias_slope(bt, st, p.bias, p.slope, t.n0, block_n, p.cout, et, EPI_THREADS * EG);
        bs = bt, ss = st;
      }
      const int H = p.H, W = p.W, cout = p.cout;

      // Output block: fetch the fp32 residual (the network input) BEFORE waiting for the accumulator.  ncu showed the
      // direct path serialising one DRAM round trip per channel behind the TMEM read (long_sb on each FADD), 10x above
      // the layer's HBM time.
      float pre[MT][4];
      if (nchw_small) {
        const int rb = t.b % res_bmod;
#pragma unroll
        for (int j = 0; j < MT; ++j) {
          if (EG == 2 && j != eg) continue;
          const int y = t.y0 + j * TH + th, x = t.x0 + tw;
          const bool valid = (y < H) && (x < W);
          const int64_t sp = static_cast<int64_t>(y) * W + x;
#pragma unroll
          for (int c = 0; c < 4; ++c)
            pre[j][c] = (valid && c < cout && p0.res_nchw != nullptr)
                            ? __ldg(p0.res_nchw + (static_cast<int64_t>(rb) * cout + c) * hw + sp) : 0.f;
        }
      }

      mbar_wait(bars + B_TFULL + acc * 8, acc_phase);
      tc_fence_after();
      if (we == 0 && lane == 0) TL_MARK_ONCE(p0, TL_ACC0, tl_first);

      // drain sub-tile j; the single-CTA loop over j is unrolled, the pair's is not
      auto drain = [&](int j) {
        if (EG == 2 && j != eg) return;   // two epilogue groups: one sub-tile each
        const int y = t.y0 + j * TH + th, x = t.x0 + tw;
        const bool valid = (y < H) && (x < W);
        const int64_t pix = (static_cast<int64_t>(t.b) * H + y) * W + x;
        const uint32_t taddr =
            tmem_base + (static_cast<uint32_t>(we * 32) << 16) + static_cast<uint32_t>(acc * MT + j) * acc_stride;
        const uint32_t rel = (EG == 2 || j == MT - 1) ? tempty + acc * 8 : 0u;
        if (nchw_small) {
          uint32_t r[16];
          tmem_ld16(taddr, r);
          tmem_ld_wait();
          if (rel != 0) {
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(rel);
          }
          if (valid) {
            const int64_t sp = static_cast<int64_t>(y) * W + x;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              if (c < cout) {
                const float a = __uint_as_float(r[c]) + bs[c];
                p0.out_nchw[(static_cast<int64_t>(t.b) * cout + c) * hw + sp] = (a > 0.f ? a : a * ss[c]) + pre[j][c];
              }
            }
          }
        } else if (staged) {
          RowMap rm;
          rm.b = t.b, rm.y0 = t.y0 + j * TH, rm.x0 = t.x0, rm.tw_shift = 3, rm.H = H, rm.W = W, rm.up = 0, rm.ky = 0, rm.kx = 0;
          epilogue_subtile_staged(ea, taddr, block_n, bs, ss, rm, we * 32, lane, t.n0, rel, stg, satm, CTAS == 2);
        } else {
          epilogue_subtile(ea, taddr, block_n, bs, ss, valid, t.b, y, x, pix, pix, t.n0, rel, satm, CTAS == 2);
        }
      };
      if constexpr (CTAS == 1) {
#pragma unroll
        for (int j = 0; j < MT; ++j) drain(j);
      } else {
#pragma unroll 1
        for (int j = 0; j < MT; ++j) drain(j);
      }
      if constexpr (CHAIN) {
        if (w.layer + 1 < prm.n_layers && w.live) {
          // publish: this warp's share of the tile is in global memory
          // (posting is never deferred past a wait: an arrival held back until the next accumulator is complete can
          // close a cycle of clusters waiting on each other's held-back arrivals in the last round of a layer)
          __threadfence();
          __syncwarp();
          if (lane == 0) red_add_gpu(prm.flags + static_cast<size_t>(w.layer) * prm.L[w.layer].num_m_tiles + w.m, 1u);
        }
      }
    }
    sat_report(sat_flag, satm);
    if (we == 0 && lane == 0) TL_MARK(p0, TL_EPI_END);
  }

  tc_fence_before();
  group_sync<CTAS>();
  if (warp == 2) {
    tc_fence_after();
    if constexpr (CTAS == 2)
      tmem_dealloc_2cta(tmem_base, static_cast<uint32_t>(prm.tmem_cols));
    else
      tmem_dealloc(tmem_base, static_cast<uint32_t>(prm.tmem_cols));
  }
#ifdef B200DN_TIMELINE
  if (threadIdx.x == 0 && p0.tl != nullptr && blockIdx.x == 0) {
    uint32_t smid;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    p0.tl[TL_SM] = smid;
    TL_MARK(p0, TL_EXIT);
  }
#endif
  if constexpr (CHAIN) {
    if (threadIdx.x == 0) {
      // the last CTA to leave closes the epoch: every poll of this launch has returned by then
      __threadfence();
      const uint32_t old = atomicAdd(prm.sync + 1, 1u);
      if (old == gridDim.x - 1) {
        prm.sync[1] = 0;
        __threadfence();
        atomicAdd(prm.sync, 1u);
      }
    }
  }
}

template <int MT, bool WRES>
__global__ void __launch_bounds__(NUM_THREADS + EPI_THREADS * (slab_epi_groups<MT, WRES>() - 1), 1)
conv3x3_slab_kernel(const __grid_constant__ KParams p) {
  conv3x3_slab_body<MT, 1, WRES>(p);
}

template <int MT>
__global__ void __launch_bounds__(NUM_THREADS, 1) conv3x3_slab2_kernel(const __grid_constant__ KParams p) {
  conv3x3_slab_body<MT, 2, false>(p);
}

template <int MT>
__global__ void __launch_bounds__(NUM_THREADS, 1) conv3x3_chain_kernel(const __grid_constant__ ChainParams c) {
  conv3x3_slab_body<MT, 2, false>(c);
}

SmemOptIn g_slab_opt_in, g_slab2_opt_in, g_chain_opt_in;

}  // namespace

int resolve_conv3x3_slab(LaunchCfg* cfg, int grid) {
  const KParams& p = cfg->p;
  B200DN_CHECK_ARG(p.wres || p.num_stages >= 2, "conv3x3 slab: W ring too small for block_n %d", p.block_n);
  B200DN_CHECK_ARG(p.num_slabs <= MAX_SLABS, "conv3x3 slab: too many slabs");
  static const void* const kernels[4] = {reinterpret_cast<const void*>(conv3x3_slab_kernel<1, false>),
                                         reinterpret_cast<const void*>(conv3x3_slab_kernel<1, true>),
                                         reinterpret_cast<const void*>(conv3x3_slab_kernel<2, false>),
                                         reinterpret_cast<const void*>(conv3x3_slab_kernel<2, true>)};
  if (int rc = ensure_max_dyn_smem(g_slab_opt_in, kernels, 4, SMEM_BYTES_SLAB,
                                   "cudaFuncSetAttribute(conv3x3_slab_kernel, smem)"))
    return rc;
  cfg->kernel = kernels[(p.mt - 1) * 2 + (p.wres ? 1 : 0)];
  cfg->grid = grid;
  cfg->threads = NUM_THREADS + ((p.mt == 2 && p.wres) ? EPI_THREADS : 0);   // second epilogue group
  cfg->smem = SMEM_BYTES_SLAB;
  cfg->cluster = 1;
  return 0;
}

int resolve_conv3x3_slab2(LaunchCfg* cfg, int grid) {
  const KParams& p = cfg->p;
  B200DN_CHECK_ARG(p.cta2 && !p.wres, "conv3x3 slab2: not a CTA-pair configuration");
  B200DN_CHECK_ARG(p.num_stages >= 2, "conv3x3 slab2: W ring too small for block_n %d", p.block_n);
  B200DN_CHECK_ARG(p.num_slabs <= MAX_SLABS, "conv3x3 slab2: too many slabs");
  B200DN_CHECK_ARG(grid >= 2 && grid % 2 == 0, "conv3x3 slab2: grid %d must be a positive multiple of 2", grid);
  static const void* const kernels[2] = {reinterpret_cast<const void*>(conv3x3_slab2_kernel<1>),
                                         reinterpret_cast<const void*>(conv3x3_slab2_kernel<2>)};
  if (int rc = ensure_max_dyn_smem(g_slab2_opt_in, kernels, 2, SMEM_BYTES_SLAB,
                                   "cudaFuncSetAttribute(conv3x3_slab2_kernel, smem)"))
    return rc;
  cfg->kernel = kernels[p.mt - 1];
  cfg->grid = grid;
  cfg->threads = NUM_THREADS;
  cfg->smem = SMEM_BYTES_SLAB;
  cfg->cluster = 2;
  return 0;
}

size_t conv_chain_workspace_bytes(const b200dn_igemm_args* a, int n) {
  // upper bound: one counter per 8 x 16 tile (MT = 1) and layer, + {epoch, exit counter}
  const size_t tiles = static_cast<size_t>(a[0].B) * cdiv(a[0].W, TW) * cdiv(a[0].H, TH);
  return (tiles * static_cast<size_t>(n > 1 ? n - 1 : 1) + 16) * sizeof(uint32_t);
}

int configure_conv_chain(const b200dn_igemm_args* a, int n, void* workspace, int flags, LaunchCfg* cfg) {
  B200DN_CHECK_ARG(a != nullptr && cfg != nullptr, "conv_chain: null argument");
  B200DN_CHECK_ARG(n >= 2 && n <= CHAIN_MAX_LAYERS, "conv_chain: %d layers (2..%d supported)", n, CHAIN_MAX_LAYERS);
  B200DN_CHECK_ARG(workspace != nullptr && (reinterpret_cast<uintptr_t>(workspace) & 15) == 0,
                   "conv_chain: workspace must be a 16-byte aligned device buffer, zero-filled once");
  ChainParams& c = cfg->c;
  memset(&c, 0, sizeof(c));
  int grid_clusters = 0;
  for (int l = 0; l < n; ++l) {
    const b200dn_igemm_args& al = a[l];
    if (al.mode != B200DN_MODE_CONV3X3 || al.out_kind != B200DN_OUT_NHWC16 || al.impl != 0 || al.block_n != 0 ||
        al.m_tiles != 0 || al.max_ctas != 0 ||
        !(al.prec == B200DN_PREC_BF16 || al.prec == B200DN_PREC_FP16)) {
      set_error("conv_chain: layer %d is not a default-configured single-plane 3x3 convolution with NHWC output", l);
      return B200DN_E_UNSUP;
    }
    B200DN_CHECK_ARG(al.B == a[0].B && al.H == a[0].H && al.W == a[0].W && al.prec == a[0].prec,
                     "conv_chain: layer %d differs from layer 0 in batch / size / precision", l);
    // a layer may overwrite nothing that it or an EARLIER layer of the chain reads as input (their tiles may still be
    // in flight): its outputs must lie beyond those input prefixes [0, cin) of the same buffer.  Later layers reading
    // them is the dependency the counters order.
    for (int j = 0; j <= l; ++j)
      B200DN_CHECK_ARG(al.out[0] != a[j].in[0] || al.out_coff >= a[j].cin,
                       "conv_chain: layer %d writes channels [%d, %d) that layer %d reads", l, al.out_coff,
                       al.out_coff + al.cout, j);
    LaunchCfg one;
    if (int rc = igemm_configure(al, &one)) return rc;
    const KParams& p = one.p;
    if (al.cout > MAX_N) {
      set_error("conv_chain: layer %d has %d outputs (bias / slopes of at most %d are staged)", l, al.cout, MAX_N);
      return B200DN_E_UNSUP;
    }
    if (!(p.cta2 && one.cluster == 2 && p.n_pairs == 1 && !p.wres)) {
      set_error("conv_chain: layer %d does not run on the CTA-pair slab kernel", l);
      return B200DN_E_UNSUP;
    }
    c.L[l] = p;
    if (l > 0 && (p.mt != c.L[0].mt || p.tiles_x != c.L[0].tiles_x || p.tiles_y != c.L[0].tiles_y ||
                  p.num_m_tiles != c.L[0].num_m_tiles || p.slab_w != c.L[0].slab_w || p.slab_bytes != c.L[0].slab_bytes)) {
      set_error("conv_chain: layers 0 and %d are tiled differently", l);
      return B200DN_E_UNSUP;
    }
    c.item_base[l + 1] = c.item_base[l] + p.num_tiles;
    c.flag_need[l] = p.num_n_tiles * (EPI_THREADS / 32);
    if (p.block_n > c.nmax) c.nmax = p.block_n;
    if (one.grid / 2 > grid_clusters) grid_clusters = one.grid / 2;
  }
  // Few tiles per layer (batch 1-2, the deep levels): every tile of layer k + 1 waits for tiles of layer k that are still
  // in flight, and a store -> fence -> counter -> poll -> TMA hand-off is no shorter than a launch boundary: measured
  // 3 % SLOWER than four launches at 2 images, 2 % faster at 32 (profiles/r02_conv_chain.txt).
  if (c.item_base[1] < 2 * grid_clusters && !(flags & B200DN_CHAIN_FORCE)) {
    set_error("conv_chain: %d pair tiles per layer on %d clusters: the layers would not overlap", c.item_base[1], grid_clusters);
    return B200DN_E_UNSUP;
  }
  for (int l = n; l < CHAIN_MAX_LAYERS; ++l) c.item_base[l + 1] = c.item_base[n];
  c.n_layers = n;
  // one ring geometry for all layers: the shallowest slab ring, the widest W stage
  int num_slabs = SLAB_MAX_SLABS, stage = 0;
  for (int l = 0; l < n; ++l) {
    if (c.L[l].num_slabs < num_slabs) num_slabs = c.L[l].num_slabs;
    if (c.L[l].stage_bytes > stage) stage = c.L[l].stage_bytes;
  }
  int num_stages = (SLAB_DATA_BYTES - num_slabs * c.L[0].slab_bytes) / stage;
  if (num_stages > MAX_STAGES) num_stages = MAX_STAGES;
  if (num_stages < 2 || num_slabs < 2) {
    set_error("conv_chain: no common ring geometry (%d slabs, %d W stages)", num_slabs, num_stages);
    return B200DN_E_UNSUP;
  }
  for (int l = 0; l < n; ++l) c.L[l].num_slabs = num_slabs, c.L[l].stage_bytes = stage, c.L[l].num_stages = num_stages;
  const int mt = c.L[0].mt;
  int cols = 32;
  while (cols < 2 * mt * c.nmax) cols <<= 1;
  if (cols > 512) {
    set_error("conv_chain: %d accumulators of %d columns do not fit TMEM", 2 * mt, c.nmax);
    return B200DN_E_UNSUP;
  }
  c.tmem_cols = cols;
  uint32_t* ws = static_cast<uint32_t*>(workspace);
  c.sync = ws;             // [0] epoch, [1] exit counter
  c.flags = ws + 16;
  static const void* const kernels[2] = {reinterpret_cast<const void*>(conv3x3_chain_kernel<1>),
                                         reinterpret_cast<const void*>(conv3x3_chain_kernel<2>)};
  if (int rc = ensure_max_dyn_smem(g_chain_opt_in, kernels, 2, SMEM_BYTES_CHAIN, "cudaFuncSetAttribute(conv3x3_chain_kernel, smem)"))
    return rc;
  // every cluster must be resident (tiles wait on tiles of other clusters)
  {
    cudaLaunchConfig_t lc;
    memset(&lc, 0, sizeof(lc));
    lc.gridDim = dim3(static_cast<unsigned>(2 * grid_clusters));
    lc.blockDim = dim3(NUM_THREADS);
    lc.dynamicSmemBytes = SMEM_BYTES_CHAIN;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2, at[0].val.clusterDim.y = 1, at[0].val.clusterDim.z = 1;
    lc.attrs = at, lc.numAttrs = 1;
    int max_clusters = 0;
    B200DN_CUDA(cudaOccupancyMaxActiveClusters(&max_clusters, kernels[mt - 1], &lc));
    if (max_clusters < 1) {
      set_error("conv_chain: no resident cluster");
      return B200DN_E_UNSUP;
    }
    if (grid_clusters > max_clusters) grid_clusters = max_clusters;
  }
#ifdef B200DN_TIMELINE
  for (int l = 0; l < n; ++l) c.L[l].tl = nullptr;
#endif
  cfg->kind = 2;
  cfg->kernel = kernels[mt - 1];
  cfg->grid = 2 * grid_clusters;
  cfg->threads = NUM_THREADS;
  cfg->smem = SMEM_BYTES_CHAIN;
  cfg->cluster = 2;
  static const bool cooperative = getenv("B200DN_CHAIN_COOP") && atoi(getenv("B200DN_CHAIN_COOP")) != 0;
  cfg->cooperative = cooperative ? 1 : 0;
  return 0;
}

}  // namespace igemm
}  // namespace b200dn

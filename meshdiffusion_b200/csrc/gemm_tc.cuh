// Persistent, warp-specialised tcgen05 implicit-GEMM kernel for sm_100a.
//
// One kernel serves every dense contraction on the score-network path (reference: nn.Conv3d call sites
// lib/diffusion/models/layers.py:118-132, NIN layers.py:573-582, attention einsums layers.py:602-606):
//
//   D[m, n] = alpha * sum_{k-steps} A_step[m, :] . B[n, kcol(step) : +KB]  (+ bias, + per-sample bias, + residual)
//
// * M indexes output voxels. An M-tile is a (bx,by,bz,bb) box of 128 voxels of the NDHWC activation tensor.
//   A tiles are fetched by TMA straight from the activation tensor as shifted 5-D boxes (zero-filled out of
//   bounds) -- no im2col buffer exists anywhere.  One A load may carry a halo along the slowest box axis so that
//   several filter taps (k-steps) reuse the same shared-memory tile through an advanced UMMA descriptor.
// * B is the packed weight matrix [N][Ktot] (K-major) whose K order is exactly the k-step order of the load
//   table, fetched by TMA as (KB x BLOCK_N) tiles.
// * Accumulators live in TMEM (2 stages), read back with tcgen05.ld by 4 epilogue warps which add bias /
//   time-embedding bias / residual, store NDHWC output and reduce per-(sample, channel) sum and sum-of-squares
//   for the GroupNorm that follows (warp-shuffle butterfly + shared + one double atomic per channel per tile).
//
// Warp roles (256 threads): w0 = TMA producer, w1 = MMA issuer, w2 = TMEM allocator, w4..7 = epilogue.
#pragma once
#include "ptx.cuh"
#include "gn_stats.cuh"

namespace mdb {

constexpr int kBlockM = 128;
constexpr int kRowBytes = 128;                       // bytes of K per row per k-step (one 128B swizzle atom)
constexpr int kAStageRows = 160;                     // 128 + up to 32 halo rows (5-tap reuse)
constexpr int kAStageBytes = kAStageRows * kRowBytes;  // 20480, multiple of 1024
constexpr int kMaxLoads = 2048;
constexpr int kMaxAMaps = 16;  // X3 doubles the maps (hi + lo parts): 8 parity sub-grids x 2
constexpr int kGemmThreads = 384;   // 4 control warps + 8 epilogue warps
constexpr int kEpiThreads = 256;

struct __align__(16) LoadEntry {
  uint8_t tmap;   // index of the A tensor map
  uint8_t nk;     // k-steps that reuse this A load
  uint8_t rows;   // rows in the A box (128 or 144)
  uint8_t jrows;  // smem row advance between consecutive k-steps of this load
  int8_t dx, dy, dz;  // coordinate offsets added to the tile origin
  uint8_t wsrc;   // (weight packer) source weight tensor
  uint16_t c0;    // channel coordinate in the A tensor
  uint16_t wc0;   // (weight packer) input-channel offset in the weight tensor; with GemmParams::b_explicit_k the
                  // K coordinate of this entry's first B tile (activation-B operands of the X3 mode)
  uint8_t tap0;   // (weight packer) tap index of k-step 0
  uint8_t tapj;   // (weight packer) tap increment per k-step
  uint16_t wpart; // (weight packer, X3) 0 = hi part bf16(w), 1 = lo part bf16(w - hi)
};
static_assert(sizeof(LoadEntry) == 16, "LoadEntry must be 16 bytes");

// A run of identical pipeline groups. One group = one shared-memory stage = one full/empty mbarrier pair:
// `epg` A boxes (1 halo box, or 2 plain boxes) and the epg*nk weight tiles they are multiplied with. All fields are
// warp-uniform kernel parameters, so the MMA warp's control flow and descriptor arithmetic never touch memory.
struct GemmSeg {
  int n_groups;
  int epg;       // load-table entries (A boxes) per group
  int nk;        // k-steps per entry
  int a_bytes;   // bytes of one A box (rows * 128) -- the TMA transaction size
  int a_stride;  // distance between the group's A boxes in the stage (multiple of 1024)
  int jbytes;    // A-descriptor advance between the k-steps of one entry (halo reuse)
  // X3 on CTA pairs: the groups of this run come in (hi, lo) couples occupying two consecutive stages -- stage k holds the
  // hi parts (A hi box, W hi tiles), stage k+1 the lo parts -- and the MMA warp issues hi*hi, hi*lo and lo*hi from the two
  // resident stages: every operand byte is fetched from L2 once for its three products (the plain K-extension form
  // fetches A hi and W hi twice).
  int x3pair;
};
constexpr int kMaxSegs = 8;

struct GemmParams {
  CUtensorMap amap[kMaxAMaps];
  CUtensorMap bmap;
  const LoadEntry* loads;
  int n_loads;
  int n_segs;
  GemmSeg segs[kMaxSegs];
  int bx, by, bz, bb;  // M-tile box (product 128)
  int X, Y, Z, Bn;     // output extents
  int tx, ty, tz, tb;  // tile counts per axis
  int n_tiles_n;
  int N;               // valid output columns
  int b_batched;       // B tensor map has a batch coordinate following the tile's sample
  int splits;          // split-K: each tile's group sequence is cut into `splits` ranges handled by different CTAs
  int total_groups;    // sum of segs[].n_groups
  float* partial;      // [splits][same layout as out] fp32 partial sums (splits > 1)
  long long split_stride;
  int dbg_flags;       // experiment switches (bit 0: cluster-scope release on the remote t_empty arrive)
  int batch_fastest;   // enumerate the batch axis first among M-tiles (residual shared by all samples stays in L2)
  int kb_elems;        // K elements per k-step (64 bf16 / 32 tf32)
  int b_explicit_k;    // B tile K coordinates come from LoadEntry::wc0 instead of the running k column
  int n_stages, stage_bytes;  // shared-memory operand ring: as many stages as fit next to the epilogue scratch
  // X3 (split bf16) epilogue: the lo parts of the output / residual rows sit this many elements behind the hi parts
  // (res1_lo_off: the second GroupNorm-backward source)
  long long out_lo_off, res_lo_off, res1_lo_off;
  // epilogue
  void* out;
  long long osx, osy, osz, osb;  // output element strides per voxel axis
  long long ocs;                 // output column stride (1 = channels contiguous; else scalar store path)
  int out_fp32;
  int round_out;  // TF32 operands: round stored activations to tf32 (rna) so downstream MMAs do not truncate them
  const float* bias;
  int bias_on_m;
  const float* rowbias;  // [Bn][rowbias_ld] per-sample bias (time embedding projection) or null
  long long rowbias_ld;
  const void* res;       // residual, same dtype as activations unless res_fp32
  long long rsx, rsy, rsz, rsb;
  int res_fp32;
  float alpha;
  long long* stats;  // [Bn][N][kStatWords] (sum, sum of squares) as split fixed-point integers (gn_stats.cuh) or null
  // ---- GroupNorm-backward fusion (GNB instantiations; training data gradients). The accumulator is dL/da of a
  // GroupNorm(+SiLU)(+dropout) output a = drop(act(gamma*xhat+beta)); `res` holds the GroupNorm INPUT x (columns
  // >= res_c0 come from res1: the second source of a channel concatenation). The epilogue stores
  // dy = da*drop*act'(y) and per-tile column partials of (sum dy, sum dy*xhat) for the GroupNorm backward.
  const void* res1;
  long long r1sx, r1sy, r1sz, r1sb;
  int res_c0;
  const float4* gnb_c;  // [Bn][N] {hsc, hsh, rs, nm}: y/2 = x*hsc + hsh, xhat = x*rs + nm
  int gnb_silu;
  int gnb_drop_thresh; float gnb_drop_scale; unsigned long long gnb_seed;
  float* gnb_part;      // [tiles_m * bb][N][2]
};

constexpr int kMaxStages = 6;
constexpr int kMaxDynSmem = 232448;  // 227 KB: the opt-in limit of dynamic shared memory per block on sm_100
template <int BLOCK_N, bool CG2>
struct GemmCfg {
  // weight tile bytes staged per CTA per k-step (a CTA pair splits the N rows of the tile between its two CTAs)
  static constexpr int kBTileBytes = BLOCK_N * kRowBytes / (CG2 ? 2 : 1);
  // The whole TMEM (512 columns) is taken: with one CTA per SM the allocation then always starts at column 0, so
  // accumulator addresses are compile-time/uniform values and the MMA issue loop needs no per-instruction R2UR.
  static constexpr int kTmemCols = 512;
  static constexpr int kStatsFloats = 24 * BLOCK_N;  // 2 x [4 warps][sum,sumsq][N] column partials + 2 x [4 segs][N] bias
  // everything but the operand ring: alignment slack, epilogue scratch, mbarriers (sized for kMaxStages), TMEM slot
  static constexpr int kFixedBytes = 1024 + kStatsFloats * 4 + (2 * kMaxStages + 4) * 8 + 16;
  // stage size / count of an op whose largest pipeline group needs `need` bytes: the ring takes whatever is left of
  // the 227 KB (more stages = more TMA bytes in flight per SM, which is what bounds the L2 -> SMEM feed rate)
  static int stage_bytes(int need) { return (need + 1023) / 1024 * 1024; }
  static int stages(int need) {
    const int n = (kMaxDynSmem - kFixedBytes) / stage_bytes(need);
    return n > kMaxStages ? kMaxStages : n;
  }
  static int smem_bytes(int need) { return kFixedBytes + stages(need) * stage_bytes(need); }
};

// dropout hash shared with the GroupNorm kernels (backward.cuh::drop_hash64)
__device__ __forceinline__ unsigned long long gn_drop_hash64(unsigned long long seed, unsigned long long idx) {
  unsigned long long z = idx + seed * 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

// D[tmem] (+)= A * B with descriptors given as their low 32 bits (start address >> 4 | LBO) and a shared constant high
// word (SBO = 1024 B, version 1, SWIZZLE_128B): all descriptor arithmetic is 32-bit adds on uniform values.
constexpr uint32_t kDescHi = (1024u >> 4) | (1u << 14) | (2u << 29);
__device__ __forceinline__ uint32_t desc_lo(uint32_t saddr) { return ((saddr & 0x3FFFFu) >> 4) | (1u << 16); }
template <bool TF32>
__device__ __forceinline__ void umma_lo(uint32_t d_tmem, uint32_t a_lo, uint32_t b_lo, uint32_t idesc, uint32_t accumulate) {
  if constexpr (TF32) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "mov.b64 da, {%1, %5};\n\tmov.b64 db, {%2, %5};\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], da, db, %3, p;\n\t}"
        :: "r"(d_tmem), "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(accumulate), "r"(kDescHi) : "memory");
  } else {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "mov.b64 da, {%1, %5};\n\tmov.b64 db, {%2, %5};\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, p;\n\t}"
        :: "r"(d_tmem), "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(accumulate), "r"(kDescHi) : "memory");
  }
}

// ---------------------------------------------------------------- CTA-pair (cta_group::2) helpers
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  // no data is published with this arrival (it only hands a TMEM stage back; tcgen05.fence orders the TMEM reads), so
  // the default cta-scope release is enough -- a cluster-scope release costs a full memory barrier per tile
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster_release(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// TMA loads whose completion bytes are credited to an mbarrier that may live in the peer CTA of the pair
__device__ __forceinline__ void tma_load_5d_cg2(const void* desc, uint32_t bar, uint32_t dst, int c0, int c1, int c2, int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
      :: "r"(dst), "l"(reinterpret_cast<uint64_t>(desc)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4) : "memory");
}
__device__ __forceinline__ void tma_load_3d_cg2(const void* desc, uint32_t bar, uint32_t dst, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4, %5}], [%2];"
      :: "r"(dst), "l"(reinterpret_cast<uint64_t>(desc)), "r"(bar), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
template <bool TF32>
__device__ __forceinline__ void umma_lo_cg2(uint32_t d_tmem, uint32_t a_lo, uint32_t b_lo, uint32_t idesc, uint32_t accumulate) {
  if constexpr (TF32) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "mov.b64 da, {%1, %5};\n\tmov.b64 db, {%2, %5};\n\t"
        "tcgen05.mma.cta_group::2.kind::tf32 [%0], da, db, %3, p;\n\t}"
        :: "r"(d_tmem), "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(accumulate), "r"(kDescHi) : "memory");
  } else {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "mov.b64 da, {%1, %5};\n\tmov.b64 db, {%2, %5};\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %3, p;\n\t}"
        :: "r"(d_tmem), "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(accumulate), "r"(kDescHi) : "memory");
  }
}
// commit of a cta_group::2 MMA batch: arrives on the mbarrier at the same offset in both CTAs of the pair
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"(static_cast<uint16_t>(3)) : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t smem_dst) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "n"(512) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(512) : "memory");
}

// CG2 = CTA pair: the two CTAs of a 2-cluster own adjacent M-tiles; the leader's single thread issues
// tcgen05.mma.cta_group::2 (M = 256) over both, each CTA stages its own A box and HALF of every weight tile, so the
// per-SM L2->SMEM traffic, the shared-memory operand reads and the MMA issue count per FLOP all drop.
// GNB: GroupNorm-backward epilogue (see GemmParams::gnb_c) -- a separate instantiation, so the inference kernels'
// code and register allocation are untouched.
// X3: split-bf16 operands (see Precision::kBF16X3): the main loop is unchanged (the three partial products are extra
// k-steps of the load table); the epilogue reads residuals and stores outputs as (hi, lo) bf16 pairs.
// M2 (CTA pairs, bf16 / tf32): every CTA owns TWO M-tiles per work item, multiplied against the SAME staged weight tiles
// (four TMEM accumulators: 2 sub-tiles x 2 stages). The kernel is bounded by operand bytes crossing L2 -> SMEM per MMA
// (ncu: profiles/r02_ncu_conv_*.txt); sharing the weight tiles between two A boxes cuts them from 3.5 KB to 2.5 KB.
template <int BLOCK_N, bool TF32, bool CG2, bool GNB = false, bool X3 = false, bool M2 = false>
__global__ void __launch_bounds__(kGemmThreads, 1) gemm_tc_kernel(const __grid_constant__ GemmParams p) {
  using Cfg = GemmCfg<BLOCK_N, CG2>;
  static_assert(!M2 || (CG2 && !X3 && BLOCK_N == 128), "M2 is built for 128-column CTA-pair kernels");
  constexpr int kSubs = M2 ? 2 : 1;
  const int NS = p.n_stages;
  const uint32_t kStageBytesRt = (uint32_t)p.stage_bytes;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  float* s_stats = reinterpret_cast<float*>(smem + NS * p.stage_bytes);
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_stats + Cfg::kStatsFloats);
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(bars + 2 * kMaxStages + 4);

  const uint32_t stage0 = smem_u32(smem);
  const uint32_t full = smem_u32(bars), empty = full + 8 * kMaxStages;
  const uint32_t t_full = empty + 8 * kMaxStages, t_empty = t_full + 16;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < kMaxAMaps; ++i) tma_prefetch_desc(&p.amap[i]);
    tma_prefetch_desc(&p.bmap);
  }
  const uint32_t rank = CG2 ? cluster_ctarank() : 0u;
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < NS; ++i) { mbar_init(full + 8 * i, 1); mbar_init(empty + 8 * i, 1); }
    // the leader's t_empty collects the epilogue warps of BOTH CTAs of a pair
    for (int i = 0; i < 2; ++i) { mbar_init(t_full + 8 * i, 1); mbar_init(t_empty + 8 * i, (CG2 ? 2 : 1) * kEpiThreads / 32); }
    fence_barrier_init();
    fence_proxy_async();
  }
  if (warp == 2) {
    if constexpr (CG2) tmem_alloc_pair(smem_u32(s_tmem));
    else tmem_alloc<Cfg::kTmemCols>(smem_u32(s_tmem));
  }
  tc_fence_before();
  if constexpr (CG2) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = 0;
  if (*s_tmem != 0) {
    if (threadIdx.x == 0) printf("mdb: unexpected TMEM base %u\n", *s_tmem);
    __trap();
  }

  const int tiles_m = p.tx * p.ty * p.tz * p.tb;
  // work items: (M-tile, N-tile) for a single CTA, (pair of adjacent M-tiles, N-tile) for a CTA pair
  const int splits = (!CG2 && p.splits > 1) ? p.splits : 1;
  const int total_tiles = (M2 ? (tiles_m + 3) / 4 : CG2 ? (tiles_m + 1) / 2 : tiles_m) * p.n_tiles_n * splits;
  const int first_tile = CG2 ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int tile_step = CG2 ? (int)(gridDim.x >> 1) : (int)gridDim.x;

  // split-K range of a work item: groups [lo, hi) of the tile's group sequence
  auto split_range = [&](int item, int& lo, int& hi) {
    const int sidx = item % splits;
    lo = (int)((long long)p.total_groups * sidx / splits);
    hi = (int)((long long)p.total_groups * (sidx + 1) / splits);
  };
  int mt_of_tile = 0;  // M-tile index of the last decoded work item (GNB partial rows)
  auto decode = [&](int tile, int& x0, int& y0, int& z0, int& b0, int& n0, int sub = 0) {
    tile /= splits;
    int nt = tile % p.n_tiles_n;
    int mt = tile / p.n_tiles_n;
    if (M2) mt = 4 * mt + 2 * (int)rank + sub;
    else if (CG2) mt = 2 * mt + (int)rank;
    mt_of_tile = mt;
    n0 = nt * BLOCK_N;
    if (mt >= tiles_m) {  // odd tile count: the pair's second CTA gets an empty tile (all loads zero-filled, no stores)
      x0 = 0; y0 = 0; z0 = 0; b0 = p.tb * p.bb;
      return;
    }
    int bt = 0;
    if (p.batch_fastest) { bt = mt % p.tb; mt /= p.tb; }
    int xt = mt % p.tx; mt /= p.tx;
    int yt = mt % p.ty; mt /= p.ty;
    int zt = mt % p.tz; mt /= p.tz;
    if (!p.batch_fastest) bt = mt;
    x0 = xt * p.bx; y0 = yt * p.by; z0 = zt * p.bz; b0 = bt * p.bb;
  };

  // Warpgroup 0 = warps 0-3 (TMA producer, MMA issuer, TMEM allocator, one idle warp); warpgroups 1-2 = the epilogue.
  // GNB only: the GroupNorm-backward epilogue is the long pole of that instantiation and it is latency-bound at 168 registers
  // (ncu source page, profiles/r02_ncu_gnb_before.txt: local-memory reloads, re-materialised S2R / LDCU, exposed constant
  // loads), so warpgroup 0 hands registers to the epilogue warpgroups: 128 x kRegsLo + 256 x kRegsHi <= 65 536. Each
  // setmaxnreg is the first instruction of its warpgroup's branch, so ptxas allocates every role with its own limit.
  constexpr int kRegsLo = 72, kRegsHi = 216;
  if (warp < 4) {
  if constexpr (GNB) setmaxnreg_dec<kRegsLo>();
  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    uint32_t st = 0, ph = 0;
    for (int tile = first_tile; tile < total_tiles; tile += tile_step) {
      int x0, y0, z0, b0, n0;
      decode(tile, x0, y0, z0, b0, n0);
      int x1 = 0, y1 = 0, z1 = 0, b1 = 0;
      if constexpr (M2) { int n1; decode(tile, x1, y1, z1, b1, n1, 1); }
      int kcol = 0, l = 0, gi = 0, g_lo, g_hi;
      split_range(tile, g_lo, g_hi);
      const int bcoord = p.b_batched ? b0 : 0;
      for (int sg = 0; sg < p.n_segs; ++sg) {
        const GemmSeg seg = p.segs[sg];
        const uint32_t group_bytes = seg.epg * (seg.a_bytes + seg.nk * Cfg::kBTileBytes);
        const uint32_t b_base = seg.epg * seg.a_stride;
        for (int g = 0; g < seg.n_groups; ++g, ++gi) {
          if (gi < g_lo || gi >= g_hi) {  // another CTA's share of this tile's K range
            kcol += seg.epg * seg.nk * p.kb_elems;
            l += seg.epg;
            continue;
          }
          // the table entries of this group are fetched before blocking on the stage
          const uint4 raw0 = __ldg(reinterpret_cast<const uint4*>(p.loads + l));
          uint4 raw1 = raw0;
          if (seg.epg > 1) raw1 = __ldg(reinterpret_cast<const uint4*>(p.loads + l + 1));
          mbar_wait(empty + 8 * st, ph ^ 1);
          if (elect_one()) {
            const uint32_t sbase = stage0 + st * kStageBytesRt;
            int kc = kcol;
            if constexpr (CG2) {
              // both CTAs credit the LEADER's full barrier; only the leader arms it (with the pair's total bytes)
              const uint32_t bar = mapa_u32(full + 8 * st, 0);
              const int nh = n0 + (int)rank * (BLOCK_N / 2);
              if constexpr (M2) {
                // one entry per group: its A box for both sub-tiles, then the weight tiles they share
                if (rank == 0) mbar_expect_tx(full + 8 * st, 2 * (2 * seg.a_bytes + seg.nk * Cfg::kBTileBytes));
                const LoadEntry& en = reinterpret_cast<const LoadEntry&>(raw0);
                tma_load_5d_cg2(&p.amap[en.tmap], bar, sbase, en.c0, x0 + en.dx, y0 + en.dy, z0 + en.dz, b0);
                tma_load_5d_cg2(&p.amap[en.tmap], bar, sbase + seg.a_stride, en.c0, x1 + en.dx, y1 + en.dy, z1 + en.dz, b1);
                for (int j = 0; j < seg.nk; ++j) {
                  tma_load_3d_cg2(&p.bmap, bar, sbase + 2 * seg.a_stride + j * Cfg::kBTileBytes, kc, nh, bcoord);
                  kc += p.kb_elems;
                }
              } else {
              if (rank == 0) mbar_expect_tx(full + 8 * st, 2 * group_bytes);
              for (int e = 0; e < seg.epg; ++e) {
                const uint4 raw = e == 0 ? raw0 : raw1;
                const LoadEntry& en = reinterpret_cast<const LoadEntry&>(raw);
                if (X3 && p.b_explicit_k) kc = en.wc0;
                tma_load_5d_cg2(&p.amap[en.tmap], bar, sbase + e * seg.a_stride, en.c0, x0 + en.dx, y0 + en.dy, z0 + en.dz, b0);
                for (int j = 0; j < seg.nk; ++j) {
                  tma_load_3d_cg2(&p.bmap, bar, sbase + b_base + (e * seg.nk + j) * Cfg::kBTileBytes, kc, nh, bcoord);
                  kc += p.kb_elems;
                }
              }
              }
            } else {
              const uint32_t bar = full + 8 * st;
              mbar_expect_tx(bar, group_bytes);
              for (int e = 0; e < seg.epg; ++e) {
                const uint4 raw = e == 0 ? raw0 : raw1;
                const LoadEntry& en = reinterpret_cast<const LoadEntry&>(raw);
                if (X3 && p.b_explicit_k) kc = en.wc0;
                tma_load_5d(&p.amap[en.tmap], bar, sbase + e * seg.a_stride, en.c0, x0 + en.dx, y0 + en.dy, z0 + en.dz, b0);
                for (int j = 0; j < seg.nk; ++j) {
                  tma_load_3d(&p.bmap, bar, sbase + b_base + (e * seg.nk + j) * Cfg::kBTileBytes, kc, n0, bcoord);
                  kc += p.kb_elems;
                }
              }
            }
          }
          __syncwarp();
          kcol += seg.epg * seg.nk * p.kb_elems;
          l += seg.epg;
          if (++st == (uint32_t)NS) { st = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == 1 && rank == 0) {
    // ------------------------------------------------------------------ MMA issuer (pair: the leader CTA only)
    constexpr uint32_t idesc = make_idesc(TF32, CG2 ? 2 * kBlockM : kBlockM, BLOCK_N);
    uint32_t st = 0, ph = 0;
    int it = 0;
    for (int tile = first_tile; tile < total_tiles; tile += tile_step, ++it) {
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      mbar_wait(t_empty + 8 * acc, acc_phase ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + acc * kSubs * BLOCK_N;
      uint32_t accumulate = 0;
      int gi = 0, g_lo, g_hi;
      split_range(tile, g_lo, g_hi);
      for (int sg = 0; sg < p.n_segs; ++sg) {
        const GemmSeg seg = p.segs[sg];
        const uint32_t b_base = seg.epg * seg.a_stride;
        if constexpr (X3 && CG2) {
          if (seg.x3pair) {
            // (hi, lo) stage couples: hi*hi as soon as the hi stage has landed, then hi*lo and lo*hi
            for (int g = 0; g < seg.n_groups; g += 2, gi += 2) {
              const uint32_t s0 = st, ph0 = ph;
              if (++st == (uint32_t)NS) { st = 0; ph ^= 1; }
              const uint32_t s1 = st, ph1 = ph;
              if (++st == (uint32_t)NS) { st = 0; ph ^= 1; }
              const uint32_t base0 = stage0 + s0 * kStageBytesRt, base1 = stage0 + s1 * kStageBytesRt;
              mbar_wait(full + 8 * s0, ph0);
              tc_fence_after();
              if (elect_one()) {
                for (int j = 0; j < seg.nk; ++j) {
                  const uint32_t a_lo = desc_lo(base0 + j * seg.jbytes);
                  const uint32_t b_lo = desc_lo(base0 + seg.a_stride + j * Cfg::kBTileBytes);
#pragma unroll
                  for (int k = 0; k < kRowBytes / 32; ++k) { umma_lo_cg2<TF32>(d_tmem, a_lo + 2 * k, b_lo + 2 * k, idesc, accumulate); accumulate = 1; }
                }
              }
              __syncwarp();
              mbar_wait(full + 8 * s1, ph1);
              tc_fence_after();
              if (elect_one()) {
                for (int j = 0; j < seg.nk; ++j) {
                  const uint32_t a0 = desc_lo(base0 + j * seg.jbytes), a1 = desc_lo(base1 + j * seg.jbytes);
                  const uint32_t b0 = desc_lo(base0 + seg.a_stride + j * Cfg::kBTileBytes);
                  const uint32_t b1 = desc_lo(base1 + seg.a_stride + j * Cfg::kBTileBytes);
#pragma unroll
                  for (int k = 0; k < kRowBytes / 32; ++k) umma_lo_cg2<TF32>(d_tmem, a0 + 2 * k, b1 + 2 * k, idesc, 1u);
#pragma unroll
                  for (int k = 0; k < kRowBytes / 32; ++k) umma_lo_cg2<TF32>(d_tmem, a1 + 2 * k, b0 + 2 * k, idesc, 1u);
                }
                umma_commit_pair(empty + 8 * s0);
                umma_commit_pair(empty + 8 * s1);
              }
              __syncwarp();
            }
            continue;
          }
        }
        for (int g = 0; g < seg.n_groups; ++g, ++gi) {
          if (gi < g_lo || gi >= g_hi) continue;
          mbar_wait(full + 8 * st, ph);
          tc_fence_after();
          if (elect_one()) {
            const uint32_t sbase = stage0 + st * kStageBytesRt;
            if constexpr (M2) {
              for (int j = 0; j < seg.nk; ++j) {
                const uint32_t b_lo = desc_lo(sbase + 2 * seg.a_stride + j * Cfg::kBTileBytes);
#pragma unroll
                for (int sub = 0; sub < 2; ++sub) {
                  const uint32_t a_lo = desc_lo(sbase + sub * seg.a_stride + j * seg.jbytes);
#pragma unroll
                  for (int k = 0; k < kRowBytes / 32; ++k)
                    umma_lo_cg2<TF32>(d_tmem + sub * BLOCK_N, a_lo + 2 * k, b_lo + 2 * k, idesc, k == 0 ? accumulate : 1u);
                }
                accumulate = 1;
              }
            } else
            for (int e = 0; e < seg.epg; ++e) {
              for (int j = 0; j < seg.nk; ++j) {
                const uint32_t a_lo = desc_lo(sbase + e * seg.a_stride + j * seg.jbytes);
                const uint32_t b_lo = desc_lo(sbase + b_base + (e * seg.nk + j) * Cfg::kBTileBytes);
#pragma unroll
                for (int k = 0; k < kRowBytes / 32; ++k) {
                  if constexpr (CG2) umma_lo_cg2<TF32>(d_tmem, a_lo + 2 * k, b_lo + 2 * k, idesc, accumulate);
                  else umma_lo<TF32>(d_tmem, a_lo + 2 * k, b_lo + 2 * k, idesc, accumulate);
                  accumulate = 1;
                }
              }
            }
            if constexpr (CG2) umma_commit_pair(empty + 8 * st); else umma_commit(empty + 8 * st);
          }
          __syncwarp();
          if (++st == (uint32_t)NS) { st = 0; ph ^= 1; }
        }
      }
      if (elect_one()) { if constexpr (CG2) umma_commit_pair(t_full + 8 * acc); else umma_commit(t_full + 8 * acc); }
      __syncwarp();
    }
  }
  } else {
    if constexpr (GNB) setmaxnreg_inc<kRegsHi>();
    // ------------------------------------------------------------------ epilogue
    // 8 epilogue warps: warp w reads TMEM lanes 32*(w%4).. (hardware rule) and owns the column chunks
    // {half, half+2, ...}; two warps per lane quarter double the latency hiding of the drain.
    const int q = warp & 3;
    const int half = (warp - 4) >> 2;
    constexpr int kChunks = BLOCK_N / 32;
    constexpr int kChunkStep = kChunks >= 2 ? 2 : 1;
    const int row = q * 32 + lane;
    const int et = threadIdx.x - 128;  // 0..255
    const int rows_per_b = p.bx * p.by * p.bz;
    const int seg = row / rows_per_b;  // which sample of the tile this row belongs to (warp-uniform by construction)
    int it = 0;
    int staged_n0 = -1, staged_b0 = -1, bias_buf = 0;
    // GNB: whether column sums are wanted is decided ONCE and pinned in a register instead of re-reading two pointers of the
    // 4 KB parameter block in front of every chunk's reduction (ncu source page, profiles/r02_ncu_gnb_after.txt: 14 % of the
    // epilogue warps' samples sat on that LDCU; by CUDA events the gain is small, 1-2 % of the GNB launches).
    int want_cols = 0;
    if constexpr (GNB) {
      want_cols = (p.stats != nullptr || p.gnb_part != nullptr) ? 1 : 0;
      asm volatile("" : "+r"(want_cols));
    }
    for (int tile = first_tile; tile < total_tiles; tile += tile_step, ++it) {
      const int acc = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
     for (int sub = 0; sub < kSubs; ++sub) {  // M2: the work item's two sub-tiles, one after the other
      const int vit = it * kSubs + sub;
      const bool last_sub = sub == kSubs - 1;
      int x0, y0, z0, b0, n0;
      decode(tile, x0, y0, z0, b0, n0, sub);
      int r = row;
      const int xl = r % p.bx; r /= p.bx;
      const int yl = r % p.by; r /= p.by;
      const int zl = r % p.bz; r /= p.bz;
      const int xg = x0 + xl, yg = y0 + yl, zg = z0 + zl, bg = b0 + r;
      const bool valid = (xg < p.X) && (yg < p.Y) && (zg < p.Z) && (bg < p.Bn);
      const long long ooff = xg * p.osx + yg * p.osy + zg * p.osz + bg * p.osb;
      const long long roff = xg * p.rsx + yg * p.rsy + zg * p.rsz + bg * p.rsb;

      // stage bias + per-sample (time-embedding) bias of this tile's columns, s_bias[seg][col] -- only when the tile's
      // (column block, first sample) differs from what is already staged (for a conv that is once per sample)
      const int bkey = p.rowbias ? b0 : 0;  // without a per-sample bias the staged values do not depend on the sample
      if (n0 != staged_n0 || bkey != staged_b0) {
        staged_n0 = n0; staged_b0 = bkey;
        bias_buf ^= 1;  // the other buffer may still be read by warps finishing the previous tile
        float* wb = s_stats + 16 * BLOCK_N + bias_buf * 4 * BLOCK_N;
        for (int i = et; i < p.bb * BLOCK_N; i += kEpiThreads) {
          const int sg = i / BLOCK_N, c = i % BLOCK_N;
          const int n = n0 + c, bgl = b0 + sg;
          float bv = 0.f;
          if (n < p.N) {
            if (p.bias && !p.bias_on_m) bv += __ldg(p.bias + n);
            if (p.rowbias && bgl < p.Bn) bv += __ldg(p.rowbias + static_cast<long long>(bgl) * p.rowbias_ld + n);
          }
          wb[i] = bv;
        }
        named_bar_sync(1, kEpiThreads);
      }
      const float* s_bias = s_stats + 16 * BLOCK_N + bias_buf * 4 * BLOCK_N;
      float* s_part = s_stats + (vit & 1) * 8 * BLOCK_N;  // column partials, double-buffered across (sub-)tiles
      // residual rows do not depend on the accumulator: fetch the first chunk while waiting for the MMAs, and every
      // next chunk while the current one is being stored, so the (L2/HBM) latency is never exposed
      uint4 rbuf[8];
      auto prefetch_res = [&](int ch) {
        const int nbp = n0 + ch * 32;
        if (!(p.res && valid && p.ocs == 1 && nbp + 32 <= p.N)) return;
        if constexpr (GNB) {
          // the GroupNorm input x: first or second source of the channel concatenation (32-column chunks never straddle)
          const bool second = p.res1 && nbp >= p.res_c0;
          const __nv_bfloat16* base = reinterpret_cast<const __nv_bfloat16*>(second ? p.res1 : p.res);
          const long long off = second ? xg * p.r1sx + yg * p.r1sy + zg * p.r1sz + bg * p.r1sb + (nbp - p.res_c0) : roff + nbp;
          const uint4* rp = reinterpret_cast<const uint4*>(base + off);
#pragma unroll
          for (int i = 0; i < 4; ++i) rbuf[i] = __ldg(rp + i);
          if constexpr (X3) {
            const uint4* rl = reinterpret_cast<const uint4*>(base + off + (second ? p.res1_lo_off : p.res_lo_off));
#pragma unroll
            for (int i = 0; i < 4; ++i) rbuf[4 + i] = __ldg(rl + i);
          }
          return;
        }
        if (TF32 || p.res_fp32) {
          const uint4* rp = reinterpret_cast<const uint4*>(reinterpret_cast<const float*>(p.res) + roff + nbp);
#pragma unroll
          for (int i = 0; i < 8; ++i) rbuf[i] = __ldg(rp + i);
        } else {
          const uint4* rp = reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(p.res) + roff + nbp);
#pragma unroll
          for (int i = 0; i < 4; ++i) rbuf[i] = __ldg(rp + i);
          if constexpr (X3) {
            const uint4* rl = reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(p.res) + roff + nbp + p.res_lo_off);
#pragma unroll
            for (int i = 0; i < 4; ++i) rbuf[4 + i] = __ldg(rl + i);
          }
        }
      };
      const int ch0 = kChunkStep == 2 ? half : 0;
      const bool active = kChunkStep == 2 || half == 0;  // BLOCK_N == 32: one chunk, the second warp of a quarter idles
      if (active) prefetch_res(ch0);
      mbar_wait(t_full + 8 * acc, acc_phase);
      tc_fence_after();
      const uint32_t t_row = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + (acc * kSubs + sub) * BLOCK_N;

#pragma unroll 1
      if (!active && last_sub) {  // nothing to drain for this warp: still release its share of the TMEM stage
        tc_fence_before();
        __syncwarp();
        if (lane == 0) { if constexpr (CG2) { if (p.dbg_flags & 1) mbar_arrive_cluster_release(mapa_u32(t_empty + 8 * acc, 0)); else mbar_arrive_cluster(mapa_u32(t_empty + 8 * acc, 0)); } else mbar_arrive(t_empty + 8 * acc); }
      }
      for (int ch = ch0; ch < kChunks && active; ch += kChunkStep) {
        uint32_t rr[32];
        tmem_ld32(t_row + ch * 32, rr);
        tmem_ld_wait();
        if (ch + kChunkStep >= kChunks && last_sub) {
          // accumulator(s) fully drained into registers: hand the TMEM stage back to the MMA warp
          tc_fence_before();
          __syncwarp();
          if (lane == 0) { if constexpr (CG2) { if (p.dbg_flags & 1) mbar_arrive_cluster_release(mapa_u32(t_empty + 8 * acc, 0)); else mbar_arrive_cluster(mapa_u32(t_empty + 8 * acc, 0)); } else mbar_arrive(t_empty + 8 * acc); }
        }
        const int nb = n0 + ch * 32;
        if (nb >= p.N) continue;  // warp-uniform
        if (splits > 1) {
          // split-K: raw fp32 partial sums; bias / residual / statistics are applied by the reduction kernel
          if (valid) {
            // (X3: ooff is in physical bf16 elements, twice the logical row pitch the fp32 partials use)
            float* pp = p.partial + (long long)(tile % splits) * p.split_stride + (X3 ? (ooff >> 1) : ooff) + nb;
            if (nb + 32 <= p.N) {
#pragma unroll
              for (int i = 0; i < 8; ++i)
                reinterpret_cast<float4*>(pp)[i] = make_float4(__uint_as_float(rr[4 * i]), __uint_as_float(rr[4 * i + 1]),
                                                               __uint_as_float(rr[4 * i + 2]), __uint_as_float(rr[4 * i + 3]));
            } else {
              for (int i = 0; i < 32; ++i) if (nb + i < p.N) pp[i] = __uint_as_float(rr[i]);
            }
          }
          continue;
        }
        const bool full = (nb + 32 <= p.N) && (p.ocs == 1);
        float v[32];
        const float mbias = (p.bias && p.bias_on_m && valid) ? __ldg(p.bias + xg) : 0.f;
        const float* sb = s_bias + (seg < 4 ? seg : 0) * BLOCK_N + ch * 32;
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(rr[i]) * p.alpha + mbias + sb[i];
        float q2[GNB ? 32 : 1];  // dy * xhat (GNB)
        if constexpr (GNB) {
          if (valid) {
            const float4* cc = p.gnb_c + static_cast<long long>(bg) * p.N + nb;
            unsigned long long hsh[8];
            if (p.gnb_drop_thresh > 0) {
              // same element index as the forward GroupNorm-apply kernel: ((b*V + voxel)*C + channel)
              const unsigned long long e4 = (unsigned long long)((((static_cast<long long>(bg) * p.Z + zg) * p.Y + yg) * p.X + xg) * p.N + nb) >> 2;
#pragma unroll
              for (int i = 0; i < 8; ++i) hsh[i] = gn_drop_hash64(p.gnb_seed, e4 + i);
            }
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              const float4 kc = __ldg(cc + i);
              const __nv_bfloat16 xb = reinterpret_cast<const __nv_bfloat16*>(rbuf)[i];
              float xv = __bfloat162float(xb);
              if constexpr (X3) xv += __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(rbuf + 4)[i]);
              float d = v[i];
              if (p.gnb_drop_thresh > 0) {
                const unsigned r16 = (unsigned)((hsh[i >> 2] >> (16 * (i & 3))) & 0xFFFFu);
                d = r16 >= (unsigned)p.gnb_drop_thresh ? d * p.gnb_drop_scale : 0.f;
              }
              if (p.gnb_silu) {
                const float h = fmaf(xv, kc.x, kc.y);
                if constexpr (X3) {
                  d *= dsilu_of_half(h);
                } else {
                  float th;
                  asm("tanh.approx.f32 %0, %1;" : "=f"(th) : "f"(h));
                  d *= fmaf(0.5f, h * fmaf(-th, th, 1.f), fmaf(0.5f, th, 0.5f));
                }
              }
              v[i] = d;
              q2[i] = d * fmaf(xv, kc.z, kc.w);
            }
          } else {
#pragma unroll
            for (int i = 0; i < 32; ++i) q2[i] = 0.f;
          }
        }
        if (!GNB && p.res && valid) {
          if (TF32 || p.res_fp32) {
            if (full) {
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                const float4 t = *reinterpret_cast<const float4*>(&rbuf[i]);
                v[4 * i] += t.x; v[4 * i + 1] += t.y; v[4 * i + 2] += t.z; v[4 * i + 3] += t.w;
              }
            } else {
              const float* rp = reinterpret_cast<const float*>(p.res) + roff + nb;
              for (int i = 0; i < 32; ++i) if (nb + i < p.N) v[i] += rp[i];
            }
          } else {
            if (full) {
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&rbuf[i]);
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                  float2 f = __bfloat1622float2(h[j]);
                  if constexpr (X3) {
                    const float2 l = __bfloat1622float2(reinterpret_cast<const __nv_bfloat162*>(&rbuf[4 + i])[j]);
                    f.x += l.x; f.y += l.y;
                  }
                  v[8 * i + 2 * j] += f.x; v[8 * i + 2 * j + 1] += f.y;
                }
              }
            } else {
              const __nv_bfloat16* rp = reinterpret_cast<const __nv_bfloat16*>(p.res) + roff + nb;
              for (int i = 0; i < 32; ++i)
                if (nb + i < p.N) v[i] += __bfloat162float(rp[i]) + (X3 ? __bfloat162float(rp[i + p.res_lo_off]) : 0.f);
            }
          }
        }
        if (ch + kChunkStep < kChunks) prefetch_res(ch + kChunkStep);  // lands while this chunk is stored / reduced
        if (valid) {
          if (TF32 || p.out_fp32) {
            float* op = reinterpret_cast<float*>(p.out) + ooff + nb;
            if (full) {
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                float4 t = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
                if (p.round_out) { t.x = to_tf32_rna(t.x); t.y = to_tf32_rna(t.y); t.z = to_tf32_rna(t.z); t.w = to_tf32_rna(t.w); }
                reinterpret_cast<float4*>(op)[i] = t;
              }
            } else {
              for (int i = 0; i < 32; ++i) if (nb + i < p.N) op[i * p.ocs] = v[i];
            }
          } else {
            __nv_bfloat16* op = reinterpret_cast<__nv_bfloat16*>(p.out) + ooff + nb;
            if (full) {
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                uint4 t;
                __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&t);
#pragma unroll
                for (int j = 0; j < 4; ++j) h[j] = __floats2bfloat162_rn(v[8 * i + 2 * j], v[8 * i + 2 * j + 1]);
                reinterpret_cast<uint4*>(op)[i] = t;
                if constexpr (X3) {  // lo parts: what the bf16 rounding of the hi parts lost
                  uint4 tl;
                  __nv_bfloat162* l = reinterpret_cast<__nv_bfloat162*>(&tl);
#pragma unroll
                  for (int j = 0; j < 4; ++j) {
                    const float2 f = __bfloat1622float2(h[j]);
                    l[j] = __floats2bfloat162_rn(v[8 * i + 2 * j] - f.x, v[8 * i + 2 * j + 1] - f.y);
                  }
                  reinterpret_cast<uint4*>(op + p.out_lo_off)[i] = tl;
                }
              }
            } else {
              for (int i = 0; i < 32; ++i)
                if (nb + i < p.N) {
                  const __nv_bfloat16 hb = __float2bfloat16(v[i]);
                  op[i * p.ocs] = hb;
                  if constexpr (X3) op[i * p.ocs + p.out_lo_off] = __float2bfloat16(v[i] - __bfloat162float(hb));
                }
            }
          }
        }
        if (GNB ? (want_cols != 0) : (p.stats != nullptr)) {  // (never reached in split-K mode)
          // Column sums over the warp's 32 rows: butterfly transpose-reduce (31 shuffles per quantity);
          // afterwards lane i holds the sum of column i.
          float s[32], ss[32];
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            const float t = valid ? v[i] : 0.f;
            s[i] = t; ss[i] = GNB ? q2[GNB ? i : 0] : t * t;
          }
#pragma unroll
          for (int off = 16; off >= 1; off >>= 1) {
            const bool hi = (lane & off) != 0;
#pragma unroll
            for (int i = 0; i < off; ++i) {
              const float send_s = hi ? s[i] : s[i + off];
              const float send_q = hi ? ss[i] : ss[i + off];
              const float keep_s = hi ? s[i + off] : s[i];
              const float keep_q = hi ? ss[i + off] : ss[i];
              s[i] = keep_s + __shfl_xor_sync(0xffffffffu, send_s, off);
              ss[i] = keep_q + __shfl_xor_sync(0xffffffffu, send_q, off);
            }
          }
          // per-warp slot, no atomics: the cross-warp sum below runs in a fixed order (deterministic results)
          s_part[(q * 2 + 0) * BLOCK_N + ch * 32 + lane] = s[0];
          s_part[(q * 2 + 1) * BLOCK_N + ch * 32 + lane] = ss[0];
        }
      }
      if constexpr (GNB) {
        if (p.gnb_part && splits == 1) {
          // per-tile column partials, one row per (M-tile, sample of the tile): summed in a fixed order by
          // gnb_tile_reduce_kernel (deterministic gradients; no atomics)
          named_bar_sync(1, kEpiThreads);
          const int warps_per_seg = rows_per_b >= 128 ? 4 : rows_per_b / 32;
          for (int i = et; i < p.bb * BLOCK_N; i += kEpiThreads) {
            const int sg = i / BLOCK_N, c = i % BLOCK_N;
            const int n = n0 + c;
            if (mt_of_tile < tiles_m && n < p.N) {
              float ts = 0.f, tq = 0.f;
              for (int w = sg * warps_per_seg; w < (sg + 1) * warps_per_seg; ++w) {
                ts += s_part[(w * 2 + 0) * BLOCK_N + c];
                tq += s_part[(w * 2 + 1) * BLOCK_N + c];
              }
              float* dst = p.gnb_part + ((static_cast<long long>(mt_of_tile) * p.bb + sg) * p.N + n) * 2;
              dst[0] = ts; dst[1] = tq;
            }
          }
        }
      }
      if (!GNB && p.stats && splits == 1) {
        // the only barrier per tile: partials of tile i+1 go to the other buffer, and a buffer is rewritten two tiles
        // later, after every warp has passed this barrier once more
        named_bar_sync(1, kEpiThreads);
        const int warps_per_seg = rows_per_b >= 128 ? 4 : rows_per_b / 32;
        for (int i = et; i < p.bb * BLOCK_N; i += kEpiThreads) {
          const int sg = i / BLOCK_N, c = i % BLOCK_N;
          const int bgl = b0 + sg, n = n0 + c;
          if (bgl < p.Bn && n < p.N) {
            float ts = 0.f, tq = 0.f;
            for (int w = sg * warps_per_seg; w < (sg + 1) * warps_per_seg; ++w) {
              ts += s_part[(w * 2 + 0) * BLOCK_N + c];
              tq += s_part[(w * 2 + 1) * BLOCK_N + c];
            }
            long long* dst = p.stats + (static_cast<long long>(bgl) * p.N + n) * kStatWords;
            stat_add(dst, ts);
            stat_add(dst + 2, tq);
          }
        }
      }
     }  // sub
    }
  }

  tc_fence_before();
  if constexpr (CG2) cluster_sync_all(); else __syncthreads();  // pair: nobody leaves while its peer may still touch it
  if (warp == 2) {
    tc_fence_after();
    if constexpr (CG2) tmem_dealloc_pair(tmem_base);
    else tmem_dealloc<Cfg::kTmemCols>(tmem_base);
  }
}

}  // namespace mdb

// tcgen05 weight-gradient kernel for sm_100a (training path: the dW half of nn.Conv3d / NIN / Linear backward,
// i.e. what autograd computes for the reference's `loss.backward()` in lib/diffusion/losses.py:104-139).
//
//   G[tap][m][n] = sum over positions p of  dY[p][m] * X[p + off(tap)][n]
//
// Both operands are NDHWC activations, so the contraction index (the voxel) is the SLOW axis of both tiles: the tiles
// are fed to the tensor cores as MN-major operands (UMMA descriptors with the 64-channel chunk stride in LBO and the
// 8-voxel group stride in SBO; a_major = b_major = 1 in the instruction descriptor) -- no transposed copy of any
// activation exists. A CTA owns ONE (Cout tile, Cin tile, tap group) and a contiguous range of voxel tiles; its up to
// three 128x128 fp32 accumulators (the ky = -1,0,+1 taps of one (kz,kx) column, served by ONE halo load of X) stay in
// TMEM for the whole range and are written once, as a split-K partial, at the end. Partials are summed in a fixed
// order by wgrad_reduce_kernel (deterministic gradients), which also scatters into the reference's OIDHW layout.
//
// Warp roles (256 threads): w0 = TMA producer, w1 = MMA issuer, w2 = TMEM allocator, w4..7 = final drain.
#pragma once
#include "gemm_tc.cuh"

namespace mdb {

constexpr int kWgThreads = 256;
constexpr int kWgStages = 3;
constexpr int kWgYChunkBytes = 128 * kRowBytes;           // 64 channels x 128 voxels
constexpr int kWgXRowsMax = 144;                          // 8 x (16 + 2 halo rows)
constexpr int kWgXChunkBytesMax = kWgXRowsMax * kRowBytes;  // 18432
constexpr int kWgStageBytes = 2 * kWgYChunkBytes + 2 * kWgXChunkBytesMax;  // 69632
constexpr int kWgSmemBytes = 1024 + kWgStages * kWgStageBytes + (2 * kWgStages + 1) * 8 + 16;
constexpr int kWgMaxGroups = 27;
constexpr int kWgMaxXMaps = 8;

struct WgradGroup {
  int8_t xmap;        // which X tensor map (stride-2 convs: the parity sub-grid of this tap)
  int8_t dx, dy, dz;  // coordinate offset of the X box relative to the dY tile origin
  int8_t ntaps;       // 1, or 3 (halo reuse along y)
  int8_t tap[3];      // output tap index of each accumulator
};
static_assert(sizeof(WgradGroup) == 8, "WgradGroup must be 8 bytes");

struct WgradParams {
  CUtensorMap ymap;
  CUtensorMap xmap[kWgMaxXMaps];
  WgradGroup groups[kWgMaxGroups];
  int n_groups;
  int bx, by, bz, bb;   // voxel tile (product 128)
  int tx, ty, tz, tb;   // voxel tile counts
  int m_tiles, n_tiles;
  int splits;           // CTAs sharing one (m tile, n tile, group): contiguous ranges of voxel tiles
  int x_chunk_bytes;    // one 64-channel X box
  int tap_shift16;      // smem advance (bytes >> 4) between the taps of a group
  int taps;             // taps of the whole operation (partial layout)
  int Mp, Np;           // padded extents (multiples of 128)
  float* partial;       // [splits][taps][Mp][Np]
  int dbg;              // bring-up switch (MDB_WG_DBG): bit 0 swaps the roles of LBO and SBO in the operand descriptors
  // X3 (split-bf16 operands): the tensor maps span the physical (hi, lo) rows, so the lo parts are the same maps at
  // channel coordinate +y_lo / +x_lo (the logical row pitches)
  int y_lo, x_lo;
};

#ifdef MDB_WGRAD_KERNEL_IMPL  // the kernel itself is compiled in wgrad_host.cu only
__device__ __forceinline__ uint32_t desc_lo_lbo(uint32_t saddr, uint32_t lbo_bytes) {
  return ((saddr & 0x3FFFFu) >> 4) | ((lbo_bytes >> 4) << 16);
}

// explicit-descriptor MMA (bring-up path only)
__device__ __forceinline__ void umma_full(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "mov.b64 da, {%1, %5};\n\tmov.b64 db, {%2, %6};\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %3, p;\n\t}"
      :: "r"(d_tmem), "r"(a_lo), "r"(b_lo), "r"(idesc), "r"(accumulate), "r"(a_hi), "r"(b_hi) : "memory");
}

// X3: G = dY_hi.X_hi + dY_hi.X_lo + dY_lo.X_hi into the same accumulators -- every voxel tile is staged three times,
// (hi, lo), (lo, hi), (hi, hi) (small terms first), with the bytes per MMA of the bf16 kernel
template <bool X3>
__global__ void __launch_bounds__(kWgThreads, 1) wgrad_tc_kernel(const __grid_constant__ WgradParams p) {
  constexpr int kPasses = X3 ? 3 : 1;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kWgStages * kWgStageBytes);
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(bars + 2 * kWgStages + 1);
  const uint32_t stage0 = smem_u32(smem);
  const uint32_t full = smem_u32(bars), empty = full + 8 * kWgStages, done = empty + 8 * kWgStages;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  // work item of this CTA
  int w = blockIdx.x;
  const int split = w % p.splits; w /= p.splits;
  const int gi = w % p.n_groups; w /= p.n_groups;
  const int nt = w % p.n_tiles;
  const int mt = w / p.n_tiles;
  const WgradGroup grp = p.groups[gi];
  const int tiles = p.tx * p.ty * p.tz * p.tb;
  const int t_lo = (int)((long long)tiles * split / p.splits);
  const int t_hi = (int)((long long)tiles * (split + 1) / p.splits);
  const int m0 = mt * 128, n0 = nt * 128;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&p.ymap);
    tma_prefetch_desc(&p.xmap[grp.xmap]);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < kWgStages; ++i) { mbar_init(full + 8 * i, 1); mbar_init(empty + 8 * i, 1); }
    mbar_init(done, 1);
    fence_barrier_init();
    fence_proxy_async();
  }
  if (warp == 2) tmem_alloc<512>(smem_u32(s_tmem));
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (*s_tmem != 0) {
    if (threadIdx.x == 0) printf("mdb: unexpected TMEM base %u\n", *s_tmem);
    __trap();
  }

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer
    uint32_t st = 0, ph = 0;
    const uint32_t bytes = 2 * kWgYChunkBytes + 2 * p.x_chunk_bytes;
    for (int it = t_lo * kPasses; it < t_hi * kPasses; ++it) {
      int r = X3 ? it / kPasses : it;
      const int pass = X3 ? it % kPasses : 0;
      const int ym = m0 + (pass == 1 ? p.y_lo : 0), xn = n0 + (pass == 0 && X3 ? p.x_lo : 0);
      const int x0 = (r % p.tx) * p.bx; r /= p.tx;
      const int y0 = (r % p.ty) * p.by; r /= p.ty;
      const int z0 = (r % p.tz) * p.bz; r /= p.tz;
      const int b0 = r * p.bb;
      mbar_wait(empty + 8 * st, ph ^ 1);
      if (elect_one()) {
        const uint32_t bar = full + 8 * st;
        const uint32_t sbase = stage0 + st * kWgStageBytes;
        mbar_expect_tx(bar, bytes);
        tma_load_5d(&p.ymap, bar, sbase, ym, x0, y0, z0, b0);
        tma_load_5d(&p.ymap, bar, sbase + kWgYChunkBytes, ym + 64, x0, y0, z0, b0);
        const uint32_t xb = sbase + 2 * kWgYChunkBytes;
        tma_load_5d(&p.xmap[grp.xmap], bar, xb, xn, x0 + grp.dx, y0 + grp.dy, z0 + grp.dz, b0);
        tma_load_5d(&p.xmap[grp.xmap], bar, xb + p.x_chunk_bytes, xn + 64, x0 + grp.dx, y0 + grp.dy, z0 + grp.dz, b0);
      }
      __syncwarp();
      if (++st == kWgStages) { st = 0; ph ^= 1; }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ MMA issuer
    constexpr uint32_t idesc = make_idesc(false, 128, 128) | (1u << 15) | (1u << 16);  // A and B MN-major
    uint32_t st = 0, ph = 0;
    for (int it = t_lo * kPasses; it < t_hi * kPasses; ++it) {
      mbar_wait(full + 8 * st, ph);
      tc_fence_after();
      if (elect_one()) {
        const uint32_t sbase = stage0 + st * kWgStageBytes;
        const uint32_t a0 = desc_lo_lbo(sbase, kWgYChunkBytes);
        const uint32_t b0 = desc_lo_lbo(sbase + 2 * kWgYChunkBytes, p.x_chunk_bytes);
        const uint32_t first = it != t_lo * kPasses ? 1u : 0u;
        if (p.dbg & 1) {
          const uint32_t hi_common = (1u << 14) | (2u << 29);
          const uint32_t a_sw = desc_lo_lbo(sbase, 1024), b_sw = desc_lo_lbo(sbase + 2 * kWgYChunkBytes, 1024);
          for (int j = 0; j < grp.ntaps; ++j)
            for (int c = 0; c < 8; ++c)
              umma_full(j * 128, a_sw + c * 128, hi_common | (kWgYChunkBytes >> 4), b_sw + j * p.tap_shift16 + c * 128,
                        hi_common | (p.x_chunk_bytes >> 4), idesc, c > 0 ? 1u : first);
        } else {
          for (int j = 0; j < grp.ntaps; ++j) {
            const uint32_t bj = b0 + j * p.tap_shift16;
#pragma unroll
            for (int c = 0; c < 8; ++c)  // 16 voxels (two 8-row swizzle atoms = 2048 B) per instruction
              umma_lo<false>(j * 128, a0 + c * 128, bj + c * 128, idesc, c > 0 ? 1u : first);
          }
        }
        umma_commit(empty + 8 * st);
      }
      __syncwarp();
      if (++st == kWgStages) { st = 0; ph ^= 1; }
    }
    if (elect_one()) umma_commit(done);
    __syncwarp();
  } else if (warp >= 4) {
    // ------------------------------------------------------------------ drain: TMEM -> fp32 partial
    mbar_wait(done, 0);
    tc_fence_after();
    const int q = warp & 3;
    const int row = q * 32 + lane;
    for (int j = 0; j < grp.ntaps; ++j) {
      float* dst = p.partial + (((long long)split * p.taps + grp.tap[j]) * p.Mp + m0 + row) * p.Np + n0;
#pragma unroll 1
      for (int ch = 0; ch < 4; ++ch) {
        uint32_t rr[32];
        tmem_ld32((static_cast<uint32_t>(q * 32) << 16) + j * 128 + ch * 32, rr);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 8; ++i)
          reinterpret_cast<float4*>(dst + ch * 32)[i] = make_float4(__uint_as_float(rr[4 * i]), __uint_as_float(rr[4 * i + 1]),
                                                                     __uint_as_float(rr[4 * i + 2]), __uint_as_float(rr[4 * i + 3]));
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc<512>(0);
  }
}

#endif  // MDB_WGRAD_KERNEL_IMPL

}  // namespace mdb

// Bandwidth-bound kernels of the training backward pass (bf16 or split-bf16 activations, fp32 parameter gradients).
// X3 (split bf16, gemm_host.h::kBF16X3): a tensor of logical row pitch ld stores [ld hi | ld lo] bf16 per voxel; the
// kernels read hi + lo as one fp32 value and write what they compute back as a (hi, lo) pair.
#include "backward.cuh"
#include "gn_stats.cuh"
#include "ptx.cuh"
#include <stdexcept>
#include <string>

namespace mdb {

#define MDB_LAUNCH_CHECK()                                                                              \
  do {                                                                                                  \
    cudaError_t _e = cudaGetLastError();                                                                \
    if (_e != cudaSuccess) throw std::runtime_error(std::string("mdb launch: ") + cudaGetErrorString(_e)); \
  } while (0)

constexpr int VEC = 8;  // bf16 elements per 16-byte vector

__device__ __forceinline__ void unpack8(const uint4& raw, float* x) {
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&raw);
#pragma unroll
  for (int j = 0; j < 4; ++j) { const float2 f = __bfloat1622float2(h[j]); x[2 * j] = f.x; x[2 * j + 1] = f.y; }
}
__device__ __forceinline__ uint4 pack8(const float* x) {
  uint4 t;
  __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&t);
#pragma unroll
  for (int j = 0; j < 4; ++j) h[j] = __floats2bfloat162_rn(x[2 * j], x[2 * j + 1]);
  return t;
}
// X3: 8 channels as hi + lo, and back (lo = what the bf16 rounding of hi lost)
__device__ __forceinline__ void unpack8x(const uint4& hi, const uint4& lo, float* x) {
  float l[VEC];
  unpack8(hi, x); unpack8(lo, l);
#pragma unroll
  for (int j = 0; j < VEC; ++j) x[j] += l[j];
}
__device__ __forceinline__ void pack8x(const float* x, uint4& hi, uint4& lo) {
  float h[VEC], r[VEC];
  hi = pack8(x);
  unpack8(hi, h);
#pragma unroll
  for (int j = 0; j < VEC; ++j) r[j] = x[j] - h[j];
  lo = pack8(r);
}

// grid.x for the staged, grid-stride kernels: the whole grid is ONE full wave of `target` = 148 x (resident blocks per
// SM) blocks -- a 608-block launch at 2 blocks/SM (296 resident) spends a third, nearly empty wave on 16 blocks.
static inline int blocks_x(long long voxels, int k, int B, int target) {
  long long gx = (voxels + (long long)k * 4 - 1) / ((long long)k * 4);
  long long want = target / B;
  if (want < 1) want = 1;
  if (gx > want) gx = want;
  return gx < 1 ? 1 : (int)gx;
}

// mean / rstd of the GroupNorm group of each of the thread's VEC channels, from the forward statistics
__device__ __forceinline__ void gn_stats_of(const GnBwdArgs& a, int b, int c, float* mean, float* rstd) {
  const int C = a.C0 + a.C1;
  const int cpg = C / a.groups;
  const double n = (double)a.voxels * cpg;
  int cur_g = -1;
  float m = 0.f, r = 0.f;
#pragma unroll
  for (int j = 0; j < VEC; ++j) {
    const int g = (c + j) / cpg;
    if (g != cur_g) {
      cur_g = g;
      StatAcc acc;
      for (int i = 0; i < cpg; ++i) {
        const int cc = g * cpg + i;
        acc.add((cc < a.C0) ? a.stats0 + ((long long)b * a.C0 + cc) * kStatWords : a.stats1 + ((long long)b * a.C1 + (cc - a.C0)) * kStatWords);
      }
      const double mm = acc.sum() / n;
      double var = acc.sumsq() / n - mm * mm;
      if (var < 0) var = 0;
      m = (float)mm;
      r = (float)(1.0 / sqrt(var + (double)a.eps));
    }
    mean[j] = m; rstd[j] = r;
  }
}

// Pass 1. Per element: h = 0.5*y straight from x (one FMA with folded constants), silu'(y) = t + 0.5*h*q with
// t = (1+tanh h)/2, q = 1 - tanh^2 h (X3: dsilu_of_half, accurate to the split operands' resolution); S2 is accumulated
// as sum(dy*x) and rebased to sum(dy*xhat) once per thread.
template <bool X3>
__global__ void __launch_bounds__(256, 2) gn_bwd_reduce_kernel(GnBwdArgs a, int cv, int k) {
  constexpr int UNROLL = X3 ? 2 : 4;  // X3: twice the bytes per voxel in flight, within the 128-register budget
  constexpr long long PP = X3 ? 2 : 1;  // physical / logical row pitch
  __shared__ float red[256 * VEC * 2];
  const int C = a.C0 + a.C1;
  const int b = blockIdx.y;
  const int cvi = threadIdx.x % cv, vl = threadIdx.x / cv;
  const int c = cvi * VEC;
  float hsc[VEC], hsh[VEC];
  {
    float mean[VEC], rstd[VEC];
    gn_stats_of(a, b, c, mean, rstd);
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      const float sc = rstd[j] * a.gamma[c + j];
      hsc[j] = 0.5f * sc;
      hsh[j] = 0.5f * fmaf(-mean[j], sc, a.beta[c + j]);
    }
  }
  const bool first = c < a.C0;
  const char* src = first ? (const char*)a.x0 + ((long long)b * a.voxels * a.ld0 * PP + c) * 2
                          : (const char*)a.x1 + ((long long)b * a.voxels * a.ld1 * PP + (c - a.C0)) * 2;
  const long long src_lo = (first ? a.ld0 : a.ld1) * 2;
  const long long src_stride = src_lo * PP;
  char* dsrc = const_cast<char*>((const char*)a.da) + ((long long)b * a.voxels * C * PP + c) * 2;
  const long long d_lo = (long long)C * 2;
  const long long d_stride = d_lo * PP;
  float s1[VEC], s2[VEC];
#pragma unroll
  for (int j = 0; j < VEC; ++j) { s1[j] = 0.f; s2[j] = 0.f; }
  const long long step = (long long)gridDim.x * k;
  for (long long v0 = (long long)blockIdx.x * k + vl; v0 < a.voxels; v0 += step * UNROLL) {
    uint4 rx[UNROLL], rd[UNROLL], rxl[X3 ? UNROLL : 1], rdl[X3 ? UNROLL : 1];
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      const long long v = v0 + u * step;
      if (v < a.voxels) {
        rx[u] = __ldg((const uint4*)(src + v * src_stride)); rd[u] = *((const uint4*)(dsrc + v * d_stride));
        if constexpr (X3) { rxl[u] = __ldg((const uint4*)(src + v * src_stride + src_lo)); rdl[u] = *((const uint4*)(dsrc + v * d_stride + d_lo)); }
      }
    }
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      const long long v = v0 + u * step;
      if (v >= a.voxels) continue;
      float x[VEC], dy[VEC];
      if constexpr (X3) { unpack8x(rx[u], rxl[u], x); unpack8x(rd[u], rdl[u], dy); }
      else { unpack8(rx[u], x); unpack8(rd[u], dy); }
      if (a.drop_thresh > 0) {
        const unsigned long long e4 = (unsigned long long)((((long long)b * a.voxels + v) * C + c) >> 2);
        const unsigned long long h0 = drop_hash64(a.seed, e4), h1 = drop_hash64(a.seed, e4 + 1);
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
          const unsigned r16 = (unsigned)(((j < 4 ? h0 : h1) >> (16 * (j & 3))) & 0xFFFFu);
          dy[j] = r16 >= (unsigned)a.drop_thresh ? dy[j] * a.drop_scale : 0.f;
        }
      }
      if (a.silu) {
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
          const float h = fmaf(x[j], hsc[j], hsh[j]);
          if constexpr (X3) {
            dy[j] *= dsilu_of_half(h);
          } else {
            float th;
            asm("tanh.approx.f32 %0, %1;" : "=f"(th) : "f"(h));
            const float q = fmaf(-th, th, 1.f);
            const float t = fmaf(0.5f, th, 0.5f);
            dy[j] *= fmaf(0.5f, h * q, t);
          }
        }
      }
#pragma unroll
      for (int j = 0; j < VEC; ++j) { s1[j] += dy[j]; s2[j] = fmaf(dy[j], x[j], s2[j]); }
      // dy replaces da in place: pass 2 then needs neither the activation derivative nor the dropout hash again
      if constexpr (X3) pack8x(dy, *((uint4*)(dsrc + v * d_stride)), *((uint4*)(dsrc + v * d_stride + d_lo)));
      else *((uint4*)(dsrc + v * d_stride)) = pack8(dy);
    }
  }
  {
    // sum(dy*xhat) = rstd*sum(dy*x) - mean*rstd*sum(dy)
    float mean[VEC], rstd[VEC];
    gn_stats_of(a, b, c, mean, rstd);
#pragma unroll
    for (int j = 0; j < VEC; ++j) s2[j] = rstd[j] * (s2[j] - mean[j] * s1[j]);
  }
#pragma unroll
  for (int j = 0; j < VEC; ++j) { red[(threadIdx.x * VEC + j) * 2] = s1[j]; red[(threadIdx.x * VEC + j) * 2 + 1] = s2[j]; }
  __syncthreads();
  if (vl == 0) {
    for (int j = 0; j < VEC; ++j) {
      float t1 = 0.f, t2 = 0.f;
      for (int l = 0; l < k; ++l) { t1 += red[((l * cv + cvi) * VEC + j) * 2]; t2 += red[((l * cv + cvi) * VEC + j) * 2 + 1]; }
      float* o = a.part + (((long long)blockIdx.x * gridDim.y + b) * C + c + j) * 2;
      o[0] = t1; o[1] = t2;
    }
  }
}

__global__ void gn_bwd_sums_kernel(const float* __restrict__ part, float* __restrict__ sums, int gx, int BC) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= BC) return;
  float t1 = 0.f, t2 = 0.f;
  for (int x = 0; x < gx; ++x) { t1 += part[((long long)x * BC + i) * 2]; t2 += part[((long long)x * BC + i) * 2 + 1]; }
  sums[2 * i] = t1; sums[2 * i + 1] = t2;
}
__global__ void gn_bwd_param_kernel(const float* __restrict__ sums, float* dgamma, float* dbeta, int B, int C, int accumulate) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  float t1 = 0.f, t2 = 0.f;
  for (int b = 0; b < B; ++b) { t1 += sums[((long long)b * C + c) * 2]; t2 += sums[((long long)b * C + c) * 2 + 1]; }
  dbeta[c] = (accumulate ? dbeta[c] : 0.f) + t1;
  dgamma[c] = (accumulate ? dgamma[c] : 0.f) + t2;
}

static void gn_launch_shape(const GnBwdArgs& a, int& cv, int& k) {
  const int C = a.C0 + a.C1;
  cv = C / VEC;
  if (cv < 1 || cv > 256 || C % VEC != 0 || a.C0 % VEC != 0) throw std::runtime_error("mdb: unsupported channel count in GroupNorm backward");
  k = 256 / cv;
}

void launch_gn_bwd_reduce(const GnBwdArgs& a, int B, cudaStream_t s) {
  int cv, k;
  gn_launch_shape(a, cv, k);
  const int C = a.C0 + a.C1;
  const int gx = blocks_x(a.voxels, k, B, 296);
  if (a.x3) gn_bwd_reduce_kernel<true><<<dim3(gx, B), cv * k, 0, s>>>(a, cv, k);
  else gn_bwd_reduce_kernel<false><<<dim3(gx, B), cv * k, 0, s>>>(a, cv, k);
  MDB_LAUNCH_CHECK();
  gn_bwd_sums_kernel<<<(B * C + 255) / 256, 256, 0, s>>>(a.part, a.sums, gx, B * C);
  MDB_LAUNCH_CHECK();
  gn_bwd_param_kernel<<<(C + 127) / 128, 128, 0, s>>>(a.sums, a.dgamma, a.dbeta, B, C, a.accumulate);
  MDB_LAUNCH_CHECK();
}

constexpr int kApplyDepth = 4;
constexpr int kApplySmem = kApplyDepth * 4 * 256 * 16;  // 64 KB (X3: twice the streams at half the depth)
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// NADD = number of addend streams (0, 1, 2): absent streams cost no instructions (GroupNorm_1 layers have none)
template <int NADD, bool X3>
__global__ void __launch_bounds__(256, X3 ? 2 : 3) gn_bwd_apply_kernel(GnBwdArgs a, int cv, int k) {
  constexpr int DEPTH = X3 ? kApplyDepth / 2 : kApplyDepth;
  constexpr int NS = X3 ? 8 : 4;        // ring slots per stage: (x, dy, add0, add1), X3: hi and lo of each
  constexpr long long PP = X3 ? 2 : 1;  // physical / logical row pitch
  __shared__ float red[256 * VEC];
  const int C = a.C0 + a.C1;
  const int b = blockIdx.y;
  const int cvi = threadIdx.x % cv, vl = threadIdx.x / cv;
  const int c = cvi * VEC;
  // dx = c1*dy - m1 - xhat*m2 (+ addends) with xhat = (x - mean)*rstd, folded to c1*dy - k0 - x*k1; `da` holds dy
  float c1[VEC], k0[VEC], k1[VEC];
  {
    float mean[VEC], rstd[VEC];
    gn_stats_of(a, b, c, mean, rstd);
    const int cpg = C / a.groups;
    const float inv_n = 1.f / ((float)a.voxels * (float)cpg);
    int cur_g = -1;
    float A = 0.f, Bq = 0.f;
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      const int gidx = (c + j) / cpg;
      if (gidx != cur_g) {
        cur_g = gidx;
        A = 0.f; Bq = 0.f;
        for (int i = 0; i < cpg; ++i) {
          const int cc = gidx * cpg + i;
          const float gm = a.gamma[cc];
          A = fmaf(gm, a.sums[((long long)b * C + cc) * 2], A);
          Bq = fmaf(gm, a.sums[((long long)b * C + cc) * 2 + 1], Bq);
        }
      }
      const float m1 = rstd[j] * A * inv_n, m2 = rstd[j] * Bq * inv_n;
      c1[j] = rstd[j] * a.gamma[c + j];
      k1[j] = rstd[j] * m2;
      k0[j] = m1 - mean[j] * rstd[j] * m2;
    }
  }
  const bool first = c < a.C0;
  const char* src = first ? (const char*)a.x0 + ((long long)b * a.voxels * a.ld0 * PP + c) * 2
                          : (const char*)a.x1 + ((long long)b * a.voxels * a.ld1 * PP + (c - a.C0)) * 2;
  const long long src_lo = (first ? a.ld0 : a.ld1) * 2;
  const long long src_stride = src_lo * PP;
  const char* dsrc = (const char*)a.da + ((long long)b * a.voxels * C * PP + c) * 2;
  const long long d_lo = (long long)C * 2;
  const long long d_stride = d_lo * PP;
  char* dst = (char*)a.dx + ((long long)b * a.voxels * C * PP + c) * 2;
  const char* p0 = NADD >= 1 ? (const char*)a.add0 + ((long long)b * a.voxels * a.add0_ld * PP + c) * 2 : nullptr;
  const char* p1 = NADD >= 2 ? (const char*)a.add1 + ((long long)b * a.voxels * a.add1_ld * PP + c) * 2 : nullptr;
  float cs[VEC];
#pragma unroll
  for (int j = 0; j < VEC; ++j) cs[j] = 0.f;
  const long long step = (long long)gridDim.x * k;
  // cp.async ring: every thread keeps kApplyDepth voxels of its own loads in flight in a private shared-memory slot
  // ring (no barriers: a thread only ever reads what it copied itself). The register-staged version of this kernel was
  // latency-bound at ~3.7 TB/s (ncu: 7 warps stalled on long-scoreboard per issue, 25-37 % occupancy); with 3 blocks/SM
  // and 4 stages there are up to 190 KB of requests outstanding per SM.
  extern __shared__ uint4 ring[];  // [DEPTH][NS streams][256 threads]
  auto slot = [&](int stage, int stream) { return ring + ((stage * NS + stream) * 256 + threadIdx.x); };
  auto issue = [&](long long vv, int stage) {
    if (vv < a.voxels) {
      cp_async16(slot(stage, 0), src + vv * src_stride);
      cp_async16(slot(stage, 1), dsrc + vv * d_stride);
      if (NADD >= 1) cp_async16(slot(stage, 2), p0 + vv * a.add0_ld * 2 * PP);
      if (NADD >= 2) cp_async16(slot(stage, 3), p1 + vv * a.add1_ld * 2 * PP);
      if constexpr (X3) {
        cp_async16(slot(stage, 4), src + vv * src_stride + src_lo);
        cp_async16(slot(stage, 5), dsrc + vv * d_stride + d_lo);
        if (NADD >= 1) cp_async16(slot(stage, 6), p0 + vv * a.add0_ld * 2 * PP + a.add0_ld * 2);
        if (NADD >= 2) cp_async16(slot(stage, 7), p1 + vv * a.add1_ld * 2 * PP + a.add1_ld * 2);
      }
    }
    cp_async_commit();
  };
  auto get = [&](int stage, int stream, float* x) {
    if constexpr (X3) unpack8x(*slot(stage, stream), *slot(stage, stream + 4), x);
    else unpack8(*slot(stage, stream), x);
  };
  long long v = (long long)blockIdx.x * k + vl;
#pragma unroll
  for (int d = 0; d < DEPTH - 1; ++d) issue(v + d * step, d);
  int stage = 0;
  for (; v < a.voxels; v += step) {
    int nst = stage + DEPTH - 1;
    if (nst >= DEPTH) nst -= DEPTH;
    issue(v + (long long)(DEPTH - 1) * step, nst);
    cp_async_wait<DEPTH - 1>();
    float x[VEC], dy[VEC], o[VEC];
    get(stage, 0, x); get(stage, 1, dy);
#pragma unroll
    for (int j = 0; j < VEC; ++j) o[j] = fmaf(-x[j], k1[j], fmaf(c1[j], dy[j], -k0[j]));
    if (NADD >= 1) {
      float e[VEC];
      get(stage, 2, e);
#pragma unroll
      for (int j = 0; j < VEC; ++j) o[j] += e[j];
    }
    if (NADD >= 2) {
      float e[VEC];
      get(stage, 3, e);
#pragma unroll
      for (int j = 0; j < VEC; ++j) o[j] += e[j];
    }
#pragma unroll
    for (int j = 0; j < VEC; ++j) cs[j] += o[j];
    if constexpr (X3) pack8x(o, *((uint4*)(dst + v * d_stride)), *((uint4*)(dst + v * d_stride + d_lo)));
    else *((uint4*)(dst + v * d_stride)) = pack8(o);
    if (++stage == DEPTH) stage = 0;
  }
  cp_async_wait<0>();
  if (a.cs_part) {  // per-(sample, channel) column sums of dx for the bias / time-embedding gradients downstream
#pragma unroll
    for (int j = 0; j < VEC; ++j) red[threadIdx.x * VEC + j] = cs[j];
    __syncthreads();
    if (vl == 0) {
      for (int j = 0; j < VEC; ++j) {
        float t = 0.f;
        for (int l = 0; l < k; ++l) t += red[(l * cv + cvi) * VEC + j];
        a.cs_part[((long long)blockIdx.x * gridDim.y + b) * C + c + j] = t;
      }
    }
  }
}

__global__ void cs_final_kernel(const float* __restrict__ part, float* __restrict__ per, int gx, int BC) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= BC) return;
  float t = 0.f;
  for (int x = 0; x < gx; ++x) t += part[(long long)x * BC + i];
  per[i] = t;
}

void launch_gn_bwd_apply(const GnBwdArgs& a, int B, cudaStream_t s) {
  int cv, k;
  gn_launch_shape(a, cv, k);
  const int C = a.C0 + a.C1;
  const int gx = blocks_x(a.voxels, k, B, 444);
  static bool configured_dev[64] = {};  // the attribute is per device
  int dev = 0;
  cudaGetDevice(&dev);
  bool& configured = configured_dev[dev < 64 ? dev : 63];
  if (!configured || dev >= 63) {
    cudaFuncSetAttribute(gn_bwd_apply_kernel<0, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kApplySmem);
    cudaFuncSetAttribute(gn_bwd_apply_kernel<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kApplySmem);
    cudaFuncSetAttribute(gn_bwd_apply_kernel<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kApplySmem);
    cudaFuncSetAttribute(gn_bwd_apply_kernel<0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kApplySmem);
    cudaFuncSetAttribute(gn_bwd_apply_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kApplySmem);
    cudaFuncSetAttribute(gn_bwd_apply_kernel<2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kApplySmem);
    configured = true;
  }
  GnBwdArgs q = a;
  if (!q.add0 && q.add1) { q.add0 = q.add1; q.add0_ld = q.add1_ld; q.add1 = nullptr; }  // streams are filled front to back
  const dim3 grid((unsigned)gx, B);
  if (q.x3) {
    if (q.add1) gn_bwd_apply_kernel<2, true><<<grid, cv * k, kApplySmem, s>>>(q, cv, k);
    else if (q.add0) gn_bwd_apply_kernel<1, true><<<grid, cv * k, kApplySmem, s>>>(q, cv, k);
    else gn_bwd_apply_kernel<0, true><<<grid, cv * k, kApplySmem, s>>>(q, cv, k);
  } else {
    if (q.add1) gn_bwd_apply_kernel<2, false><<<grid, cv * k, kApplySmem, s>>>(q, cv, k);
    else if (q.add0) gn_bwd_apply_kernel<1, false><<<grid, cv * k, kApplySmem, s>>>(q, cv, k);
    else gn_bwd_apply_kernel<0, false><<<grid, cv * k, kApplySmem, s>>>(q, cv, k);
  }
  MDB_LAUNCH_CHECK();
  if (a.cs_part) {
    cs_final_kernel<<<(B * C + 255) / 256, 256, 0, s>>>(a.cs_part, a.cs_per, gx, B * C);
    MDB_LAUNCH_CHECK();
  }
}

// ------------------------------------------------------------------ fused path: constants for the GEMM epilogue, tile reduce
__global__ void gn_consts_kernel(GnBwdArgs a, float4* __restrict__ out, int B) {
  const int C = a.C0 + a.C1;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * C) return;
  const int b = i / C, c = i % C;
  const int cpg = C / a.groups, g = c / cpg;
  StatAcc acc;
  for (int j = 0; j < cpg; ++j) {
    const int cc = g * cpg + j;
    acc.add((cc < a.C0) ? a.stats0 + ((long long)b * a.C0 + cc) * kStatWords : a.stats1 + ((long long)b * a.C1 + (cc - a.C0)) * kStatWords);
  }
  const double n = (double)a.voxels * cpg;
  const double mm = acc.sum() / n;
  double var = acc.sumsq() / n - mm * mm;
  if (var < 0) var = 0;
  const float mean = (float)mm, rstd = (float)(1.0 / sqrt(var + (double)a.eps));
  const float sc = rstd * a.gamma[c];
  out[i] = make_float4(0.5f * sc, 0.5f * fmaf(-mean, sc, a.beta[c]), rstd, -mean * rstd);
}
void launch_gn_consts(const GnBwdArgs& a, float* consts4, int B, cudaStream_t s) {
  const int C = a.C0 + a.C1;
  gn_consts_kernel<<<(B * C + 255) / 256, 256, 0, s>>>(a, reinterpret_cast<float4*>(consts4), B);
  MDB_LAUNCH_CHECK();
}

// grid (ceil(C/32), B), block (32, 8): lane y sums tiles y, y+8, ... in order; the 8 lane sums are added in order
__global__ void gnb_tile_reduce_kernel(const float* __restrict__ part, float* __restrict__ sums, int T, int bb, int C) {
  __shared__ float red[8][32][2];
  const int b = blockIdx.y, c = blockIdx.x * 32 + threadIdx.x;
  const long long row0 = (long long)(b / bb) * T;
  const int sg = b % bb;
  float t1 = 0.f, t2 = 0.f;
  if (c < C) {
    for (int t = threadIdx.y; t < T; t += 8) {
      const float2 v = *reinterpret_cast<const float2*>(part + (((row0 + t) * bb + sg) * C + c) * 2);
      t1 += v.x; t2 += v.y;
    }
  }
  red[threadIdx.y][threadIdx.x][0] = t1; red[threadIdx.y][threadIdx.x][1] = t2;
  __syncthreads();
  if (threadIdx.y == 0 && c < C) {
    t1 = 0.f; t2 = 0.f;
    for (int l = 0; l < 8; ++l) { t1 += red[l][threadIdx.x][0]; t2 += red[l][threadIdx.x][1]; }
    sums[((long long)b * C + c) * 2] = t1; sums[((long long)b * C + c) * 2 + 1] = t2;
  }
}
void launch_gnb_tile_reduce(const GnBwdArgs& a, const float* tile_part, int T, int bb, int B, cudaStream_t s) {
  const int C = a.C0 + a.C1;
  gnb_tile_reduce_kernel<<<dim3((C + 31) / 32, B), dim3(32, 8), 0, s>>>(tile_part, a.sums, T, bb, C);
  MDB_LAUNCH_CHECK();
  gn_bwd_param_kernel<<<(C + 127) / 128, 128, 0, s>>>(a.sums, a.dgamma, a.dbeta, B, C, a.accumulate);
  MDB_LAUNCH_CHECK();
}

// ------------------------------------------------------------------ column sums (bias / time-embedding gradients)
template <bool X3>
__global__ void __launch_bounds__(256) colsum_kernel(ColsumArgs a, int cv, int k) {
  constexpr int UNROLL = 4;
  constexpr long long PP = X3 ? 2 : 1;
  __shared__ float red[256 * VEC];
  const int b = blockIdx.y;
  const int cvi = threadIdx.x % cv, vl = threadIdx.x / cv;
  const int c = cvi * VEC;
  const char* src = (const char*)a.t + ((long long)b * a.voxels * a.ld * PP + c) * 2;
  float s1[VEC];
#pragma unroll
  for (int j = 0; j < VEC; ++j) s1[j] = 0.f;
  const long long step = (long long)gridDim.x * k;
  for (long long v0 = (long long)blockIdx.x * k + vl; v0 < a.voxels; v0 += step * UNROLL) {
    uint4 r[UNROLL], rl[X3 ? UNROLL : 1];
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      const long long v = v0 + u * step;
      r[u] = make_uint4(0, 0, 0, 0);
      if constexpr (X3) rl[u] = make_uint4(0, 0, 0, 0);
      if (v < a.voxels) {
        r[u] = __ldg((const uint4*)(src + v * a.ld * 2 * PP));
        if constexpr (X3) rl[u] = __ldg((const uint4*)(src + v * a.ld * 2 * PP + a.ld * 2));
      }
    }
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      float x[VEC];
      if constexpr (X3) unpack8x(r[u], rl[u], x);
      else unpack8(r[u], x);
#pragma unroll
      for (int j = 0; j < VEC; ++j) s1[j] += x[j];
    }
  }
#pragma unroll
  for (int j = 0; j < VEC; ++j) red[threadIdx.x * VEC + j] = s1[j];
  __syncthreads();
  if (vl == 0) {
    for (int j = 0; j < VEC; ++j) {
      float t = 0.f;
      for (int l = 0; l < k; ++l) t += red[(l * cv + cvi) * VEC + j];
      a.part[((long long)blockIdx.x * gridDim.y + b) * a.C + c + j] = t;
    }
  }
}
// grid = ceil(C / 32) blocks of (32 channels x 8 lanes): a lane sums the block partials x = lane, lane + 8, ... of one
// (sample, channel), the 8 lane sums are added in lane order, samples in batch order -- deterministic, and 8x the
// parallelism of one thread per channel walking all gx * B partials (27 us per launch before)
__global__ void __launch_bounds__(256) colsum_final_kernel(ColsumArgs a, int gx, int B) {
  __shared__ float red[8][32];
  const int c = blockIdx.x * 32 + threadIdx.x;
  float tot = 0.f;
  for (int b = 0; b < B; ++b) {
    float t = 0.f;
    if (c < a.C) {
      if (a.from_per) { if (threadIdx.y == 0) t = a.part[(long long)b * a.from_ld + c]; }
      else for (int x = threadIdx.y; x < gx; x += 8) t += a.part[((long long)x * B + b) * a.C + c];
    }
    red[threadIdx.y][threadIdx.x] = t;
    __syncthreads();
    if (threadIdx.y == 0 && c < a.C) {
      float sb = 0.f;
      for (int l = 0; l < 8; ++l) sb += red[l][threadIdx.x];
      if (a.per) a.per[(long long)b * a.per_ld + c] = sb;
      tot += sb;
    }
    __syncthreads();
  }
  if (threadIdx.y == 0 && c < a.C) {
    if (a.total0) a.total0[c] = (a.accumulate ? a.total0[c] : 0.f) + tot;
    if (a.total1) a.total1[c] = (a.accumulate ? a.total1[c] : 0.f) + tot;
    if (a.total2) a.total2[c] = (a.accumulate ? a.total2[c] : 0.f) + tot;
  }
}
void launch_colsum(const ColsumArgs& a, int B, cudaStream_t s) {
  if (a.from_per) {  // the producer already left per-sample sums ([B][from_ld] floats): only the batch sum remains
    ColsumArgs c = a;
    c.part = const_cast<float*>(a.from_per);
    colsum_final_kernel<<<(a.C + 31) / 32, dim3(32, 8), 0, s>>>(c, 1, B);
    MDB_LAUNCH_CHECK();
    return;
  }
  const int cv = a.C / VEC;
  if (cv < 1 || cv > 256 || a.C % VEC != 0) throw std::runtime_error("mdb: unsupported channel count in colsum");
  const int k = 256 / cv;
  const int gx = blocks_x(a.voxels, k, B, 592);
  if (a.x3) colsum_kernel<true><<<dim3(gx, B), cv * k, 0, s>>>(a, cv, k);
  else colsum_kernel<false><<<dim3(gx, B), cv * k, 0, s>>>(a, cv, k);
  MDB_LAUNCH_CHECK();
  colsum_final_kernel<<<(a.C + 31) / 32, dim3(32, 8), 0, s>>>(a, gx, B);
  MDB_LAUNCH_CHECK();
}

// ------------------------------------------------------------------ resampling data movement
static inline int grid_for(long long work_items, int threads) {
  long long b = (work_items + threads - 1) / threads;
  const long long cap = 148LL * 8;
  if (b > cap) b = cap;
  return b < 1 ? 1 : (int)b;
}

__global__ void zero_stuff2x_kernel(const uint4* __restrict__ dy, uint4* __restrict__ z, int B, int R, int cv) {
  const int R2 = 2 * R;
  const long long total = (long long)B * R2 * R2 * R2 * cv;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    long long r = i;
    const int c = (int)(r % cv); r /= cv;
    const int xo = (int)(r % R2); r /= R2;
    const int yo = (int)(r % R2); r /= R2;
    const int zo = (int)(r % R2); r /= R2;
    uint4 v = make_uint4(0, 0, 0, 0);
    if ((xo & yo & zo & 1) != 0) v = __ldg(dy + ((((long long)r * R + (zo >> 1)) * R + (yo >> 1)) * R + (xo >> 1)) * cv + c);
    z[i] = v;
  }
}
void launch_zero_stuff2x(const void* dy, void* z, int B, int R, int C, cudaStream_t s) {
  const int cv = C / VEC;
  const long long total = (long long)B * 8 * R * R * R * cv;
  zero_stuff2x_kernel<<<grid_for(total, 256), 256, 0, s>>>((const uint4*)dy, (uint4*)z, B, R, cv);
  MDB_LAUNCH_CHECK();
}

// X3: rows of cv hi vectors then cv lo vectors
template <bool X3>
__global__ void downsum2x_kernel(const uint4* __restrict__ dup, uint4* __restrict__ dx, int B, int R, int cv) {
  constexpr int PP = X3 ? 2 : 1;
  const int R2 = 2 * R;
  const long long total = (long long)B * R * R * R * cv;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    long long r = i;
    const int c = (int)(r % cv); r /= cv;
    const int xo = (int)(r % R); r /= R;
    const int yo = (int)(r % R); r /= R;
    const int zo = (int)(r % R); r /= R;
    float acc[VEC];
#pragma unroll
    for (int j = 0; j < VEC; ++j) acc[j] = 0.f;
    for (int dz = 0; dz < 2; ++dz)
      for (int dyy = 0; dyy < 2; ++dyy)
        for (int dxx = 0; dxx < 2; ++dxx) {
          float t[VEC];
          const uint4* sp = dup + ((((long long)r * R2 + 2 * zo + dz) * R2 + 2 * yo + dyy) * R2 + 2 * xo + dxx) * cv * PP + c;
          if constexpr (X3) unpack8x(__ldg(sp), __ldg(sp + cv), t);
          else unpack8(__ldg(sp), t);
#pragma unroll
          for (int j = 0; j < VEC; ++j) acc[j] += t[j];
        }
    if constexpr (X3) {
      uint4* dp = dx + (i - c) * PP + c;
      pack8x(acc, dp[0], dp[cv]);
    } else {
      dx[i] = pack8(acc);
    }
  }
}
void launch_downsum2x(const void* dup, void* dx, int B, int R, int C, int x3, cudaStream_t s) {
  const int cv = C / VEC;
  const long long total = (long long)B * R * R * R * cv;
  if (x3) downsum2x_kernel<true><<<grid_for(total, 256), 256, 0, s>>>((const uint4*)dup, (uint4*)dx, B, R, cv);
  else downsum2x_kernel<false><<<grid_for(total, 256), 256, 0, s>>>((const uint4*)dup, (uint4*)dx, B, R, cv);
  MDB_LAUNCH_CHECK();
}

// n = logical vectors per sample; X3: rows of cv hi vectors then cv lo vectors
template <bool X3>
__global__ void batch_sum_kernel(const uint4* __restrict__ t, uint4* __restrict__ out, int B, long long n, int cv) {
  constexpr int PP = X3 ? 2 : 1;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const long long pi = X3 ? (i / cv) * 2 * cv + i % cv : i;  // physical index of the (hi) vector
    float acc[VEC];
#pragma unroll
    for (int j = 0; j < VEC; ++j) acc[j] = 0.f;
    for (int b = 0; b < B; ++b) {
      float x[VEC];
      const uint4* sp = t + (long long)b * n * PP + pi;
      if constexpr (X3) unpack8x(__ldg(sp), __ldg(sp + cv), x);
      else unpack8(__ldg(sp), x);
#pragma unroll
      for (int j = 0; j < VEC; ++j) acc[j] += x[j];
    }
    if constexpr (X3) pack8x(acc, out[pi], out[pi + cv]);
    else out[i] = pack8(acc);
  }
}
void launch_batch_sum(const void* t, void* out, int B, long long VC, int C, int x3, cudaStream_t s) {
  const long long n = VC / VEC;
  if (x3) batch_sum_kernel<true><<<grid_for(n, 256), 256, 0, s>>>((const uint4*)t, (uint4*)out, B, n, C / VEC);
  else batch_sum_kernel<false><<<grid_for(n, 256), 256, 0, s>>>((const uint4*)t, (uint4*)out, B, n, C / VEC);
  MDB_LAUNCH_CHECK();
}

__global__ void __launch_bounds__(1024) rowsum_nc_kernel(const float* __restrict__ t, float* out, int B, int C, long long V, int accumulate) {
  __shared__ float red[32];
  const int c = blockIdx.x;
  float acc = 0.f;
  for (int b = 0; b < B; ++b) {
    const float* p = t + ((long long)b * C + c) * V;
    for (long long v = threadIdx.x; v < V; v += blockDim.x) acc += __ldg(p + v);
  }
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tot = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) tot += red[w];
    out[c] = (accumulate ? out[c] : 0.f) + tot;
  }
}
void launch_rowsum_nc(const float* t, float* out, int B, int C, long long V, int accumulate, cudaStream_t s) {
  rowsum_nc_kernel<<<C, 1024, 0, s>>>(t, out, B, C, V, accumulate);
  MDB_LAUNCH_CHECK();
}

// ------------------------------------------------------------------ attention softmax backward (layers.py:604)
template <bool X3>  // X3: P and dS rows are [L hi | L lo] bf16 (the same bytes as L fp32 slots)
__global__ void __launch_bounds__(256) softmax_bwd_rows_kernel(const float* __restrict__ P, float* __restrict__ dP, long long rows, int L) {
  __shared__ float red[8];
  for (long long row = blockIdx.x; row < rows; row += gridDim.x) {
    const __nv_bfloat16* p = reinterpret_cast<const __nv_bfloat16*>(P + row * L);
    float* d = dP + row * L;
    float pv[16], dv[16];
    float dot = 0.f;
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const int i = threadIdx.x + j * 256;
      pv[j] = i < L ? __bfloat162float(p[i]) + (X3 ? __bfloat162float(p[L + i]) : 0.f) : 0.f;
      dv[j] = i < L ? d[i] : 0.f;
      dot = fmaf(pv[j], dv[j], dot);
    }
    for (int o = 16; o; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = dot;
    __syncthreads();  // also: every thread has read its dP values before anyone overwrites the row
    dot = 0.f;
    for (int w = 0; w < 8; ++w) dot += red[w];
    __syncthreads();
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const int i = threadIdx.x + j * 256;
      if (i < L) {
        const float ds = pv[j] * (dv[j] - dot);
        const __nv_bfloat16 hb = __float2bfloat16(ds);
        reinterpret_cast<__nv_bfloat16*>(d)[i] = hb;
        if (X3) reinterpret_cast<__nv_bfloat16*>(d)[L + i] = __float2bfloat16(ds - __bfloat162float(hb));
      }
    }
  }
}
void launch_softmax_bwd_rows(const float* P, float* dP, long long rows, int L, int x3, cudaStream_t s) {
  if (L > 16 * 256) throw std::runtime_error("mdb: softmax row too long");
  const int grid = (int)(rows < 148LL * 16 ? rows : 148LL * 16);
  if (x3) softmax_bwd_rows_kernel<true><<<grid, 256, 0, s>>>(P, dP, rows, L);
  else softmax_bwd_rows_kernel<false><<<grid, 256, 0, s>>>(P, dP, rows, L);
  MDB_LAUNCH_CHECK();
}

// ------------------------------------------------------------------ small fp32 linear-layer gradients (time embedding)
__global__ void outer_sum_kernel(const float* __restrict__ dy, long long dy_ld, const float* __restrict__ x, long long x_ld,
                                 float* dW, float* db, int B, int N, int K, int accumulate) {
  const long long total = (long long)N * K;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int n = (int)(i / K), k = (int)(i % K);
    float acc = 0.f;
    for (int b = 0; b < B; ++b) acc = fmaf(dy[b * dy_ld + n], x[b * x_ld + k], acc);
    dW[i] = (accumulate ? dW[i] : 0.f) + acc;
    if (k == 0 && db) {
      float t = 0.f;
      for (int b = 0; b < B; ++b) t += dy[b * dy_ld + n];
      db[n] = (accumulate ? db[n] : 0.f) + t;
    }
  }
}
void launch_outer_sum(const float* dy, long long dy_ld, const float* x, long long x_ld, float* dW, float* db, int B, int N, int K,
                      int accumulate, cudaStream_t s) {
  outer_sum_kernel<<<grid_for((long long)N * K, 256), 256, 0, s>>>(dy, dy_ld, x, x_ld, dW, db, B, N, K, accumulate);
  MDB_LAUNCH_CHECK();
}

__global__ void dense_bwd_input_kernel(const float* __restrict__ dy, long long dy_ld, const float* __restrict__ W, float* __restrict__ dx,
                                       int B, int N, int K) {
  const int b = blockIdx.y;
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= K) return;
  float acc = 0.f;
  for (int n = 0; n < N; ++n) acc = fmaf(dy[b * dy_ld + n], __ldg(W + (long long)n * K + k), acc);
  dx[(long long)b * K + k] = acc;
}
void launch_dense_bwd_input(const float* dy, long long dy_ld, const float* W, float* dx, int B, int N, int K, cudaStream_t s) {
  dense_bwd_input_kernel<<<dim3((K + 127) / 128, B), 128, 0, s>>>(dy, dy_ld, W, dx, B, N, K);
  MDB_LAUNCH_CHECK();
}

__device__ __forceinline__ float sigmoid_f(float x) { return 1.f / (1.f + __expf(-x)); }

// One block per sample. Recomputes emb -> t1 -> h1 -> t2 (elementwise.cu temb_kernel), then
// dt2 = dact * silu'(t2), dh1 = W1^T dt2, dt1 = dh1 * silu'(t1).
__global__ void temb_bwd_kernel(const float* __restrict__ labels, const float* __restrict__ w0, const float* __restrict__ b0,
                                const float* __restrict__ w1, const float* __restrict__ b1, const float* __restrict__ dact,
                                float* __restrict__ dt2, float* __restrict__ h1o, float* __restrict__ dt1, float* __restrict__ embo, int nf) {
  extern __shared__ float sm[];
  const int H = 4 * nf;
  float* emb = sm;          // nf
  float* t1 = sm + nf;      // H
  float* h1 = t1 + H;       // H
  float* d2 = h1 + H;       // H
  const int b = blockIdx.x;
  const int half = nf / 2;
  const float t = labels[b];
  for (int i = threadIdx.x; i < nf; i += blockDim.x) {
    const int k = i < half ? i : i - half;
    const float coef = logf(10000.f) / (float)(half - 1);
    const float f = expf((float)k * -coef);
    const float arg = t * f;
    emb[i] = i < half ? sinf(arg) : cosf(arg);
    embo[(long long)b * nf + i] = emb[i];
  }
  __syncthreads();
  for (int n = threadIdx.x; n < H; n += blockDim.x) {
    float acc = b0[n];
    for (int k = 0; k < nf; ++k) acc += w0[(long long)n * nf + k] * emb[k];
    t1[n] = acc;
    const float sg = sigmoid_f(acc);
    h1[n] = acc * sg;
    h1o[(long long)b * H + n] = h1[n];
  }
  __syncthreads();
  for (int n = threadIdx.x; n < H; n += blockDim.x) {
    float acc = b1[n];
    for (int k = 0; k < H; ++k) acc += w1[(long long)n * H + k] * h1[k];
    const float sg = sigmoid_f(acc);
    const float d = dact[(long long)b * H + n] * sg * (1.f + acc * (1.f - sg));
    d2[n] = d;
    dt2[(long long)b * H + n] = d;
  }
  __syncthreads();
  for (int k = threadIdx.x; k < H; k += blockDim.x) {
    float acc = 0.f;
    for (int n = 0; n < H; ++n) acc = fmaf(d2[n], __ldg(w1 + (long long)n * H + k), acc);
    const float sg = sigmoid_f(t1[k]);
    dt1[(long long)b * H + k] = acc * sg * (1.f + t1[k] * (1.f - sg));
  }
}
void launch_temb_bwd(const float* labels, const float* w0, const float* b0, const float* w1, const float* b1, const float* dact,
                     float* dt2, float* h1, float* dt1, float* emb, int B, int nf, cudaStream_t s) {
  temb_bwd_kernel<<<B, 256, (nf + 12 * nf) * sizeof(float), s>>>(labels, w0, b0, w1, b1, dact, dt2, h1, dt1, emb, nf);
  MDB_LAUNCH_CHECK();
}

}  // namespace mdb

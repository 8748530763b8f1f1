#include "elementwise.cuh"
#include "backward.cuh"
#include "gn_stats.cuh"
#include <curand_kernel.h>
#include <stdexcept>
#include <string>

namespace mdb {

#define MDB_LAUNCH_CHECK()                                                                              \
  do {                                                                                                  \
    cudaError_t _e = cudaGetLastError();                                                                \
    if (_e != cudaSuccess) throw std::runtime_error(std::string("mdb launch: ") + cudaGetErrorString(_e)); \
  } while (0)

static inline int grid_for(long long work_items, int threads) {
  long long b = (work_items + threads - 1) / threads;
  const long long cap = 148LL * 8;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return (int)b;
}

__device__ __forceinline__ float round_tf32_rna(float x) {
  uint32_t u;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(x));
  return __uint_as_float(u);
}
// x * sigmoid(x) = x / (1 + 2^(-x log2 e)) in five instructions: ex2.approx + rcp.approx (each ~1 ulp; the IEEE division and
// __frcp_rn expand to a MUFU plus Newton steps -- ncu showed the bf16x3 GroupNorm pass issue-bound at 32 instructions per
// element with them, profiles/r02_ncu_norm_act_x3.txt)
__device__ __forceinline__ float silu_f(float x) {
  float e, r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * -1.4426950408889634f));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.f + e));
  return x * r;
}
// x*sigmoid(x) = 0.5x(1 + tanh(x/2)) with the single-MUFU tanh.approx (rel. error 2^-11: below bf16 resolution, not
// below the 2^-16 of a split-bf16 pair, so only the bf16 kernels use it); halves the MUFU pressure of the bf16
// GroupNorm+SiLU pass, which otherwise co-limits with HBM bandwidth.
__device__ __forceinline__ float silu_fast(float x) {
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(0.5f * x));
  const float h = 0.5f * x;
  return fmaf(h, t, h);
}

// ------------------------------------------------------------------ GroupNorm finalize
// nn.GroupNorm(32, C, eps=1e-6) statistics (layers.py:589,652,660; ddpm_res64.py:120): biased variance over
// (C/32) channels x voxels. Channel sums arrive from the producing GEMM's epilogue as split fixed-point integer pairs (gn_stats.cuh)
// (integer atomics commute, so the statistics -- and with them the whole forward pass -- are bitwise reproducible).
__global__ void gn_finalize_kernel(GnFinalizeArgs a) {
  const int b = blockIdx.x;
  const int C = a.C0 + a.C1;
  const int cpg = C / a.groups;
  for (int g = threadIdx.x; g < a.groups; g += blockDim.x) {
    StatAcc acc;
    for (int i = 0; i < cpg; ++i) {
      const int c = g * cpg + i;
      acc.add((c < a.C0) ? a.stats0 + ((long long)b * a.C0 + c) * kStatWords
                         : a.stats1 + ((long long)b * a.C1 + (c - a.C0)) * kStatWords);
    }
    const double s = acc.sum(), ss = acc.sumsq();
    const double n = a.count_per_channel * cpg;
    const double mean = s / n;
    double var = ss / n - mean * mean;
    if (var < 0) var = 0;
    const float rstd = (float)(1.0 / sqrt(var + (double)a.eps));
    for (int i = 0; i < cpg; ++i) {
      const int c = g * cpg + i;
      const float sc = a.gamma[c] * rstd;
      a.scale[(long long)b * C + c] = sc;
      a.shift[(long long)b * C + c] = a.beta[c] - (float)mean * sc;
    }
  }
}
void launch_gn_finalize(const GnFinalizeArgs& a, int B, cudaStream_t s) {
  gn_finalize_kernel<<<B, 32, 0, s>>>(a);
  MDB_LAUNCH_CHECK();
}

// ------------------------------------------------------------------ GroupNorm apply (+SiLU), concat-aware
// blockIdx.y = sample. Every thread owns ONE 16-byte channel vector for the whole kernel (block = k voxels x C/VEC
// vectors): its scale/shift live in registers, its source pointer is selected once, and the loop body is
// load -> fma -> silu -> store with 4 voxels in flight. No div/mod or table lookups in the loop: the kernel is
// HBM-bound instead of issue-bound.
// MODE: 0 = bf16, 1 = tf32 (fp32 storage), 2 = split bf16 (X3: a channel vector is a 16-byte hi part and a 16-byte lo
// part one logical row apart, on the input as on the output)
template <int MODE>
__global__ void __launch_bounds__(256, MODE == 1 ? 4 : 3) norm_act_kernel(NormActArgs a, int cv, int k) {
  constexpr bool TF32 = MODE == 1;
  constexpr bool X3 = MODE == 2;
  constexpr int VEC = TF32 ? 4 : 8;  // 16 bytes
  constexpr int UNROLL = 4;
  const int C = a.C0 + a.C1;
  const int b = blockIdx.y;
  const int cvi = threadIdx.x % cv, vl = threadIdx.x / cv;
  const int c = cvi * VEC;
  float sc[VEC], sh[VEC];
  if (a.stats0) {
    // GroupNorm finalize fused into the prologue: each thread derives mean / rstd of the group(s) of ITS channels from
    // the per-channel sums the producing GEMM left behind (cpg channels x 2 values, L2-resident) -- 80 fewer launches
    const int cpg = C / a.groups;
    const double n = (double)a.voxels * cpg;
    int cur_g = -1;
    float mean = 0.f, rstd = 0.f;
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      const int ch = c + j, g = ch / cpg;
      if (g != cur_g) {
        cur_g = g;
        StatAcc acc;
        for (int i = 0; i < cpg; ++i) {
          const int cc = g * cpg + i;
          acc.add((cc < a.C0) ? a.stats0 + ((long long)b * a.C0 + cc) * kStatWords
                              : a.stats1 + ((long long)b * a.C1 + (cc - a.C0)) * kStatWords);
        }
        const double m = acc.sum() / n;
        double var = acc.sumsq() / n - m * m;
        if (var < 0) var = 0;
        mean = (float)m;
        rstd = (float)(1.0 / sqrt(var + (double)a.eps));
      }
      sc[j] = a.gamma[ch] * rstd;
      sh[j] = a.beta[ch] - mean * sc[j];
    }
  } else {
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      sc[j] = a.scale[(long long)b * C + c + j];
      sh[j] = a.shift[(long long)b * C + c + j];
    }
  }
  const int es = TF32 ? 4 : 2;
  constexpr int PARTS = X3 ? 2 : 1;
  const bool first = c < a.C0;
  const char* src = first ? (const char*)a.x0 + ((long long)b * a.voxels * a.ld0 * PARTS + c) * es
                          : (const char*)a.x1 + ((long long)b * a.voxels * a.ld1 * PARTS + (c - a.C0)) * es;
  const long long src_stride = (first ? a.ld0 : a.ld1) * es * PARTS;  // bytes per voxel
  const long long src_lo = (first ? a.ld0 : a.ld1) * es;              // X3: hi -> lo distance in bytes
  char* dst = (char*)a.y + ((long long)b * a.voxels * C * PARTS + c) * es;
  const long long dst_stride = (long long)C * es * PARTS;
  const long long dst_lo = (long long)C * es;
  const long long step = (long long)gridDim.x * k;
  for (long long v0 = (long long)blockIdx.x * k + vl; v0 < a.voxels; v0 += step * UNROLL) {
    uint4 raw[UNROLL], rawl[X3 ? UNROLL : 1];
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      const long long v = v0 + u * step;
      if (v < a.voxels) {
        raw[u] = __ldg((const uint4*)(src + v * src_stride));
        if constexpr (X3) rawl[u] = __ldg((const uint4*)(src + v * src_stride + src_lo));
      }
    }
#pragma unroll
    for (int u = 0; u < UNROLL; ++u) {
      const long long v = v0 + u * step;
      if (v >= a.voxels) continue;
      float x[VEC];
      if (TF32) {
        const float* f = (const float*)&raw[u];
#pragma unroll
        for (int j = 0; j < VEC; ++j) x[j] = f[j];
      } else {
        const __nv_bfloat162* h = (const __nv_bfloat162*)&raw[u];
#pragma unroll
        for (int j = 0; j < 4; ++j) { float2 f = __bfloat1622float2(h[j]); x[2 * j] = f.x; x[2 * j + 1] = f.y; }
        if constexpr (X3) {
          const __nv_bfloat162* l = (const __nv_bfloat162*)&rawl[u];
#pragma unroll
          for (int j = 0; j < 4; ++j) { float2 f = __bfloat1622float2(l[j]); x[2 * j] += f.x; x[2 * j + 1] += f.y; }
        }
      }
#pragma unroll
      for (int j = 0; j < VEC; ++j) {
        float y = fmaf(x[j], sc[j], sh[j]);
        if (a.silu) y = MODE == 0 ? silu_fast(y) : silu_f(y);
        x[j] = y;
      }
      if (!TF32 && a.drop_thresh > 0) {  // (training plans: bf16 and split bf16; same element index in both)
        const unsigned long long e4 = (unsigned long long)((((long long)b * a.voxels + v) * C + c) >> 2);
        const unsigned long long h0 = drop_hash64(a.seed, e4), h1 = drop_hash64(a.seed, e4 + 1);
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
          const unsigned r16 = (unsigned)(((j < 4 ? h0 : h1) >> (16 * (j & 3))) & 0xFFFFu);
          x[j] = r16 >= (unsigned)a.drop_thresh ? x[j] * a.drop_scale : 0.f;
        }
      }
      if (TF32) {
        *((float4*)(dst + v * dst_stride)) =
            make_float4(round_tf32_rna(x[0]), round_tf32_rna(x[1]), round_tf32_rna(x[2]), round_tf32_rna(x[3]));
      } else {
        uint4 t;
        __nv_bfloat162* h = (__nv_bfloat162*)&t;
#pragma unroll
        for (int j = 0; j < 4; ++j) h[j] = __floats2bfloat162_rn(x[2 * j], x[2 * j + 1]);
        *((uint4*)(dst + v * dst_stride)) = t;
        if constexpr (X3) {
          uint4 tl;
          __nv_bfloat162* l = (__nv_bfloat162*)&tl;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float2 f = __bfloat1622float2(h[j]);
            l[j] = __floats2bfloat162_rn(x[2 * j] - f.x, x[2 * j + 1] - f.y);
          }
          *((uint4*)(dst + v * dst_stride + dst_lo)) = tl;
        }
      }
    }
  }
}
void launch_norm_act(const NormActArgs& a, int B, cudaStream_t s) {
  const int vec = a.tf32 == 1 ? 4 : 8;
  const int C = a.C0 + a.C1;
  const int cv = C / vec;
  if (cv > 256 || cv < 1 || a.C0 % vec != 0) throw std::runtime_error("mdb: unsupported channel count in norm_act");
  const int k = 256 / cv;  // voxels per block pass
  const int threads = cv * k;
  long long gx = (a.voxels + (long long)k * 4 - 1) / ((long long)k * 4);
  const long long cap = (148LL * 8 + B - 1) / B;
  if (gx > cap) gx = cap;
  if (gx < 1) gx = 1;
  dim3 grid((unsigned)gx, (unsigned)B);
  if (a.tf32 == 1) norm_act_kernel<1><<<grid, threads, 0, s>>>(a, cv, k);
  else if (a.tf32 == 2) norm_act_kernel<2><<<grid, threads, 0, s>>>(a, cv, k);
  else norm_act_kernel<0><<<grid, threads, 0, s>>>(a, cv, k);
  MDB_LAUNCH_CHECK();
}

// ------------------------------------------------------------------ nearest 2x upsample (layers.py:620)
__global__ void upsample2x_kernel(const uint4* __restrict__ x, uint4* __restrict__ y, int B, int Z, int Y, int X, int cv) {
  const long long total = (long long)B * (2 * Z) * (2 * Y) * (2 * X) * cv;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    long long r = i;
    const int c = (int)(r % cv); r /= cv;
    const int xo = (int)(r % (2 * X)); r /= (2 * X);
    const int yo = (int)(r % (2 * Y)); r /= (2 * Y);
    const int zo = (int)(r % (2 * Z)); r /= (2 * Z);
    const long long src = ((((long long)r * Z + (zo >> 1)) * Y + (yo >> 1)) * X + (xo >> 1)) * cv + c;
    y[i] = __ldg(x + src);
  }
}
void launch_upsample2x(const void* x, void* y, int B, int Z, int Y, int X, int C, int tf32, cudaStream_t s) {
  const int cv = C / (tf32 ? 4 : 8);
  const long long total = (long long)B * 8 * Z * Y * X * cv;
  upsample2x_kernel<<<grid_for(total, 256), 256, 0, s>>>((const uint4*)x, (uint4*)y, B, Z, Y, X, cv);
  MDB_LAUNCH_CHECK();
}

// ------------------------------------------------------------------ stem im2col
// One block per (sample, z, group of YB y-rows): the k x (k+YB-1) input rows it needs are staged in shared memory once
// (a warp per row, no per-element div/mod), then every thread emits 16-byte vectors of the [voxel][Kpad] operand
// matrix (column = cin*k^3 + tap) through a per-column slab-offset table.
constexpr int kIm2colYB = 4;
template <int MODE>  // 0 bf16, 1 tf32, 2 split bf16 (row = [Kpad hi | Kpad lo])
__global__ void __launch_bounds__(256) im2col_kernel(const float* __restrict__ x, void* __restrict__ a, int Cin, int R, int k, int Kpad) {
  constexpr bool TF32 = MODE == 1;
  constexpr bool X3 = MODE == 2;
  constexpr int VEC = TF32 ? 4 : 8;
  constexpr int YB = kIm2colYB;
  extern __shared__ float slab[];  // [Cin][k][k+YB-1][R + 2*pad]
  const int pad = k / 2, W = R + 2 * pad, T = k * k * k, KH = k + YB - 1;
  const int yblocks = R / YB;
  const int y0 = (blockIdx.x % yblocks) * YB, z0 = (blockIdx.x / yblocks) % R, b = blockIdx.x / (yblocks * R);
  const long long V = (long long)R * R * R;
  const int n_rows = Cin * k * KH;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int row = warp; row < n_rows; row += 8) {
    const int khh = row % KH, kd = (row / KH) % k, ci = row / (KH * k);
    const int zi = z0 + kd - pad, yi = y0 + khh - pad;
    const bool row_ok = zi >= 0 && zi < R && yi >= 0 && yi < R;
    const float* src = x + ((long long)b * Cin + ci) * V + ((long long)zi * R + yi) * R;
    for (int xw = lane; xw < W; xw += 32) {
      const int xi = xw - pad;
      slab[row * W + xw] = (row_ok && xi >= 0 && xi < R) ? __ldg(src + xi) : 0.f;
    }
  }
  int* coloff = reinterpret_cast<int*>(slab + n_rows * W);
  for (int col = threadIdx.x; col < Kpad; col += blockDim.x) {
    int off = -1;
    if (col < Cin * T) {
      const int ci = col / T, tap = col % T;
      const int kd = tap / (k * k), kh = (tap / k) % k, kw = tap % k;
      off = ((ci * k + kd) * KH + kh) * W + kw;
    }
    coloff[col] = off;
  }
  __syncthreads();
  const int kv = Kpad / VEC;
  for (int yb = 0; yb < YB; ++yb) {
    const long long row0 = (((long long)b * R + z0) * R + y0 + yb) * R;
    const int ybase = yb * W;
    for (int i = threadIdx.x; i < R * kv; i += blockDim.x) {
      const int xo = i / kv, col0 = (i - xo * kv) * VEC;
      float v[VEC];
#pragma unroll
      for (int j = 0; j < VEC; ++j) {
        const int off = coloff[col0 + j];
        v[j] = off >= 0 ? slab[off + ybase + xo] : 0.f;
      }
      if (TF32) {
        *((float4*)((float*)a + (row0 + xo) * Kpad + col0)) =
            make_float4(round_tf32_rna(v[0]), round_tf32_rna(v[1]), round_tf32_rna(v[2]), round_tf32_rna(v[3]));
      } else {
        uint4 t;
        __nv_bfloat162* h = (__nv_bfloat162*)&t;
#pragma unroll
        for (int j = 0; j < 4; ++j) h[j] = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
        if constexpr (X3) {
          uint4 tl;
          __nv_bfloat162* l = (__nv_bfloat162*)&tl;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float2 f = __bfloat1622float2(h[j]);
            l[j] = __floats2bfloat162_rn(v[2 * j] - f.x, v[2 * j + 1] - f.y);
          }
          *((uint4*)((__nv_bfloat16*)a + (row0 + xo) * 2 * Kpad + col0)) = t;
          *((uint4*)((__nv_bfloat16*)a + (row0 + xo) * 2 * Kpad + Kpad + col0)) = tl;
        } else {
          *((uint4*)((__nv_bfloat16*)a + (row0 + xo) * Kpad + col0)) = t;
        }
      }
    }
  }
}
void launch_im2col(const float* x, void* a, int B, int Cin, int R, int k, int Kpad, int tf32, cudaStream_t s) {
  if (R % kIm2colYB != 0) throw std::runtime_error("mdb: im2col needs a grid size divisible by 4");
  const size_t smem = (size_t)Cin * k * (k + kIm2colYB - 1) * (R + 2 * (k / 2)) * sizeof(float) + (size_t)Kpad * sizeof(int);
  static bool configured[64] = {};  // per device
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev >= 64 || !configured[dev]) {
    cudaFuncSetAttribute(im2col_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);
    cudaFuncSetAttribute(im2col_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);
    cudaFuncSetAttribute(im2col_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);
    if (dev < 64) configured[dev] = true;
  }
  if (smem > 100 * 1024) throw std::runtime_error("mdb: im2col slab too large");
  const unsigned grid = (unsigned)(B * R * (R / kIm2colYB));
  if (tf32 == 1) im2col_kernel<1><<<grid, 256, smem, s>>>(x, a, Cin, R, k, Kpad);
  else if (tf32 == 2) im2col_kernel<2><<<grid, 256, smem, s>>>(x, a, Cin, R, k, Kpad);
  else im2col_kernel<0><<<grid, 256, smem, s>>>(x, a, Cin, R, k, Kpad);
  MDB_LAUNCH_CHECK();
}

// ------------------------------------------------------------------ row softmax (layers.py:604)
template <int MODE>  // 0 bf16, 1 tf32, 2 split bf16: hi parts in the first L bf16 of the row, lo parts in the next L
__global__ void softmax_rows_kernel(float* __restrict__ s, long long rows, int L) {
  constexpr bool TF32 = MODE == 1;
  __shared__ float red[32];
  for (long long row = blockIdx.x; row < rows; row += gridDim.x) {
    float* p = s + row * L;
    float vals[16];  // L <= 16 * blockDim.x; fully unrolled so the array stays in registers
    float m = -INFINITY;
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const int i = threadIdx.x + j * 256;
      vals[j] = i < L ? p[i] : -INFINITY;
      m = fmaxf(m, vals[j]);
    }
    for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
    __syncthreads();
    m = red[0];
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) m = fmaxf(m, red[w]);
    __syncthreads();
    float sum = 0.f;
#pragma unroll
    for (int j = 0; j < 16; ++j) { vals[j] = __expf(vals[j] - m); sum += vals[j]; }
    for (int o = 16; o; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = sum;
    __syncthreads();
    sum = 0.f;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) sum += red[w];
    const float inv = 1.f / sum;
    __syncthreads();  // every thread has consumed its fp32 logits before anyone overwrites the row
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const int i = threadIdx.x + j * 256;
      if (i < L) {
        if (TF32) p[i] = round_tf32_rna(vals[j] * inv);
        else {
          const float pv = vals[j] * inv;
          const __nv_bfloat16 hb = __float2bfloat16(pv);
          ((__nv_bfloat16*)p)[i] = hb;
          if (MODE == 2) ((__nv_bfloat16*)p)[L + i] = __float2bfloat16(pv - __bfloat162float(hb));
        }
      }
    }
  }
}
void launch_softmax_rows(float* s, long long rows, int L, int tf32, cudaStream_t st) {
  if (L > 16 * 256) throw std::runtime_error("mdb: softmax row too long");
  const int grid = (int)(rows < 148LL * 16 ? rows : 148LL * 16);
  if (tf32 == 1) softmax_rows_kernel<1><<<grid, 256, 0, st>>>(s, rows, L);
  else if (tf32 == 2) softmax_rows_kernel<2><<<grid, 256, 0, st>>>(s, rows, L);
  else softmax_rows_kernel<0><<<grid, 256, 0, st>>>(s, rows, L);
  MDB_LAUNCH_CHECK();
}

// ------------------------------------------------------------------ V transpose: out[b][c][v] = in[b][v][c0+c]
template <typename T>
__global__ void transpose_vc_kernel(const T* __restrict__ in, long long ld, int c0, T* __restrict__ out, int V, int C, long long ldo) {
  __shared__ T tile[32][33];
  const int b = blockIdx.z;
  const int v0 = blockIdx.x * 32, cb = blockIdx.y * 32;
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    const int v = v0 + j, c = cb + threadIdx.x;
    if (v < V && c < C) tile[j][threadIdx.x] = in[((long long)b * V + v) * ld + c0 + c];
  }
  __syncthreads();
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    const int c = cb + j, v = v0 + threadIdx.x;
    if (v < V && c < C) out[((long long)b * C + c) * ldo + v] = tile[threadIdx.x][j];
  }
}
// bf16 fast path: 64x64 tiles, two elements (4 bytes) per thread on both the read and the write side, so every warp
// moves full 128-byte rows (the 32x32 / 2-byte version touched half-used sectors in both directions)
__global__ void __launch_bounds__(256) transpose_vc_bf16x2_kernel(const __nv_bfloat16* __restrict__ in, long long ld, int c0,
                                                                  __nv_bfloat16* __restrict__ out, int V, int C, long long ldo) {
  __shared__ __nv_bfloat16 tile[64][66];
  const int b = blockIdx.z;
  const int v0 = blockIdx.x * 64, cb = blockIdx.y * 64;
  const int tx = threadIdx.x, ty = threadIdx.y;
  for (int j = ty; j < 64; j += 8) {
    const int v = v0 + j, c = cb + 2 * tx;
    if (v < V && c + 1 < C) {
      const __nv_bfloat162 t = *reinterpret_cast<const __nv_bfloat162*>(in + ((long long)b * V + v) * ld + c0 + c);
      tile[j][2 * tx] = t.x; tile[j][2 * tx + 1] = t.y;
    }
  }
  __syncthreads();
  for (int j = ty; j < 64; j += 8) {
    const int c = cb + j, v = v0 + 2 * tx;
    if (c < C && v + 1 < V) {
      __nv_bfloat162 t;
      t.x = tile[2 * tx][j]; t.y = tile[2 * tx + 1][j];
      *reinterpret_cast<__nv_bfloat162*>(out + ((long long)b * C + c) * ldo + v) = t;
    }
  }
}

void launch_transpose_vc(const void* in, long long ld, int c0, void* out, int B, int V, int C, int tf32, cudaStream_t s,
                         long long ld_out) {
  const long long ldo = ld_out ? ld_out : V;
  if (!tf32 && V % 64 == 0 && C % 64 == 0 && ld % 2 == 0 && c0 % 2 == 0 && ldo % 2 == 0) {
    dim3 grid(V / 64, C / 64, B), block(32, 8);
    transpose_vc_bf16x2_kernel<<<grid, block, 0, s>>>((const __nv_bfloat16*)in, ld, c0, (__nv_bfloat16*)out, V, C, ldo);
    MDB_LAUNCH_CHECK();
    return;
  }
  dim3 grid((V + 31) / 32, (C + 31) / 32, B), block(32, 8);
  if (tf32) transpose_vc_kernel<float><<<grid, block, 0, s>>>((const float*)in, ld, c0, (float*)out, V, C, ldo);
  else transpose_vc_kernel<__nv_bfloat16><<<grid, block, 0, s>>>((const __nv_bfloat16*)in, ld, c0, (__nv_bfloat16*)out, V, C, ldo);
  MDB_LAUNCH_CHECK();
}
void launch_transpose_vc_rows(const void* in, long long ld, int c0, void* out, int B, int V, int C, int x3, cudaStream_t s) {
  if (!x3) { launch_transpose_vc(in, ld, c0, out, B, V, C, 0, s); return; }
  launch_transpose_vc(in, 2 * ld, c0, out, B, V, C, 0, s, 2LL * V);
  launch_transpose_vc(in, 2 * ld, (int)ld + c0, (__nv_bfloat16*)out + V, B, V, C, 0, s, 2LL * V);
}

// ------------------------------------------------------------------ time embedding MLP
// get_timestep_embedding (layers.py:542-556): half = nf/2, freq_k = exp(-ln(1e4) * k / (half-1)), [sin, cos];
// then Linear(nf,4nf) -> SiLU -> Linear(4nf,4nf) (ddpm_res64.py:132-136); ResnetBlockDDPM applies act(temb) before
// Dense_0 (layers.py:680), so act(temb) is what every consumer needs and is what we store.
__global__ void temb_kernel(const float* __restrict__ labels, const float* __restrict__ w0, const float* __restrict__ b0,
                            const float* __restrict__ w1, const float* __restrict__ b1, float* __restrict__ out, int nf) {
  extern __shared__ float sm[];
  float* emb = sm;            // nf
  float* h1 = sm + nf;        // 4nf
  const int b = blockIdx.x;
  const int half = nf / 2;
  const float t = labels[b];
  for (int i = threadIdx.x; i < nf; i += blockDim.x) {
    const int k = i < half ? i : i - half;
    const float coef = logf(10000.f) / (float)(half - 1);
    const float f = expf((float)k * -coef);
    const float arg = t * f;
    emb[i] = i < half ? sinf(arg) : cosf(arg);
  }
  __syncthreads();
  const int H = 4 * nf;
  for (int n = threadIdx.x; n < H; n += blockDim.x) {
    float acc = b0[n];
    for (int k = 0; k < nf; ++k) acc += w0[(long long)n * nf + k] * emb[k];
    h1[n] = silu_f(acc);
  }
  __syncthreads();
  for (int n = threadIdx.x; n < H; n += blockDim.x) {
    float acc = b1[n];
    for (int k = 0; k < H; ++k) acc += w1[(long long)n * H + k] * h1[k];
    out[(long long)b * H + n] = silu_f(acc);
  }
}
void launch_temb(const float* labels, const float* w0, const float* b0, const float* w1, const float* b1, float* out,
                 int B, int nf, cudaStream_t s) {
  temb_kernel<<<B, 256, 5 * nf * sizeof(float), s>>>(labels, w0, b0, w1, b1, out, nf);
  MDB_LAUNCH_CHECK();
}

__global__ void dense_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ bias,
                             float* __restrict__ out, int B, int K, int N) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  for (int o = warp; o < B * N; o += nwarps) {
    const int b = o / N, n = o % N;
    float acc = 0.f;
    for (int k = lane; k < K; k += 32) acc += w[(long long)n * K + k] * x[(long long)b * K + k];
    for (int s = 16; s; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
    if (lane == 0) out[(long long)b * N + n] = acc + bias[n];
  }
}
void launch_dense(const float* x, const float* w, const float* bias, float* out, int B, int K, int N, cudaStream_t s) {
  dense_kernel<<<grid_for((long long)B * N * 32, 256), 256, 0, s>>>(x, w, bias, out, B, K, N);
  MDB_LAUNCH_CHECK();
}

// ------------------------------------------------------------------ head conv phase 2: tap shift-sum (Cout == 4)
template <bool PFP32>
__global__ void __launch_bounds__(256) tap_shift_sum_kernel(const void* __restrict__ P, long long ldp, const float* __restrict__ bias,
                                                           float* __restrict__ out, int R, int k) {
  const int pad = k / 2;
  const long long V = (long long)R * R * R;
  const int b = blockIdx.y;
  for (long long v = blockIdx.x * (long long)blockDim.x + threadIdx.x; v < V; v += (long long)gridDim.x * blockDim.x) {
    const int x = (int)(v % R), y = (int)((v / R) % R), z = (int)(v / ((long long)R * R));
    float acc0 = bias[0], acc1 = bias[1], acc2 = bias[2], acc3 = bias[3];
    int tap = 0;
    for (int dz = -pad; dz <= pad; ++dz)
      for (int dy = -pad; dy <= pad; ++dy)
        for (int dx = -pad; dx <= pad; ++dx, ++tap) {
          const int zz = z + dz, yy = y + dy, xx = x + dx;
          if ((unsigned)zz >= (unsigned)R || (unsigned)yy >= (unsigned)R || (unsigned)xx >= (unsigned)R) continue;
          const long long row = ((long long)b * V + ((long long)zz * R + yy) * R + xx) * ldp + tap * 4;
          if (PFP32) {
            const float4 t = __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(P) + row));
            acc0 += t.x; acc1 += t.y; acc2 += t.z; acc3 += t.w;
          } else {
            const uint2 t = __ldg(reinterpret_cast<const uint2*>(reinterpret_cast<const __nv_bfloat16*>(P) + row));
            const float2 f0 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&t.x));
            const float2 f1 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&t.y));
            acc0 += f0.x; acc1 += f0.y; acc2 += f1.x; acc3 += f1.y;
          }
        }
    float* o = out + (long long)b * 4 * V + v;
    o[0] = acc0; o[V] = acc1; o[2 * V] = acc2; o[3 * V] = acc3;
  }
}
void launch_tap_shift_sum(const void* P, long long ldp, int p_fp32, const float* bias, float* out, int B, int R, int k,
                          int Cout, cudaStream_t s) {
  if (Cout != 4) throw std::runtime_error("mdb: tap_shift_sum supports 4 output channels");
  const long long V = (long long)R * R * R;
  long long gx = (V + 255) / 256;
  const long long cap = (148LL * 16 + B - 1) / B;
  if (gx > cap) gx = cap;
  dim3 grid((unsigned)gx, (unsigned)B);
  if (p_fp32) tap_shift_sum_kernel<true><<<grid, 256, 0, s>>>(P, ldp, bias, out, R, k);
  else tap_shift_sum_kernel<false><<<grid, 256, 0, s>>>(P, ldp, bias, out, R, k);
  MDB_LAUNCH_CHECK();
}

// ------------------------------------------------------------------ split-K reduction
// blockIdx.y = sample, blockIdx.x = chunk of voxels; thread = output channel (coalesced rows). Each thread owns a
// channel for its chunk, so its statistics are accumulated in a fixed order (deterministic) and published with one
// integer atomic per (block, channel).
template <int MODE>  // 0 bf16, 1 tf32, 2 split bf16 (out / res rows are [N hi | N lo])
__global__ void __launch_bounds__(256) split_reduce_kernel(SplitReduceArgs a, int vchunk) {
  constexpr bool TF32 = MODE == 1;
  const int b = blockIdx.y;
  const long long v0 = (long long)blockIdx.x * vchunk;
  const long long v1 = v0 + vchunk < a.voxels ? v0 + vchunk : a.voxels;
  for (int n = threadIdx.x; n < a.N; n += blockDim.x) {
    float add = a.bias ? a.bias[n] : 0.f;
    if (a.rowbias) add += a.rowbias[(long long)b * a.rowbias_ld + n];
    float s1 = 0.f, s2 = 0.f;
    for (long long v = v0; v < v1; ++v) {
      const long long idx = ((long long)b * a.voxels + v) * a.N + n;
      float acc = add;
      for (int sp = 0; sp < a.splits; ++sp) acc += a.partial[sp * a.split_stride + idx];
      if (a.res) {
        const long long ridx = (long long)b * a.res_batch_stride + v * a.N + n;
        if (MODE == 2) {
          const __nv_bfloat16* rp = (const __nv_bfloat16*)a.res + 2 * ((long long)b * a.res_batch_stride + v * a.N) + n;
          acc += __bfloat162float(rp[0]) + __bfloat162float(rp[a.N]);
        } else {
          acc += TF32 ? ((const float*)a.res)[ridx] : __bfloat162float(((const __nv_bfloat16*)a.res)[ridx]);
        }
      }
      s1 += acc; s2 += acc * acc;
      if (TF32) ((float*)a.out)[idx] = round_tf32_rna(acc);
      else if (MODE == 2) {
        __nv_bfloat16* op = (__nv_bfloat16*)a.out + 2 * (idx - n) + n;
        const __nv_bfloat16 hb = __float2bfloat16(acc);
        op[0] = hb;
        op[a.N] = __float2bfloat16(acc - __bfloat162float(hb));
      }
      else ((__nv_bfloat16*)a.out)[idx] = __float2bfloat16(acc);
    }
    if (a.stats) {
      long long* dst = a.stats + ((long long)b * a.N + n) * kStatWords;
      stat_add(dst, s1);
      stat_add(dst + 2, s2);
    }
  }
}
void launch_split_reduce(const SplitReduceArgs& a, int B, cudaStream_t s) {
  const int vchunk = 8;
  dim3 grid((unsigned)((a.voxels + vchunk - 1) / vchunk), (unsigned)B);
  const int threads = a.N < 256 ? ((a.N + 31) / 32) * 32 : 256;
  if (a.tf32 == 1) split_reduce_kernel<1><<<grid, threads, 0, s>>>(a, vchunk);
  else if (a.tf32 == 2) split_reduce_kernel<2><<<grid, threads, 0, s>>>(a, vchunk);
  else split_reduce_kernel<0><<<grid, threads, 0, s>>>(a, vchunk);
  MDB_LAUNCH_CHECK();
}

__global__ void add_vec_kernel(const float* a, const float* b, float* out, int n) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) out[i] = a[i] + (b ? b[i] : 0.f);
}
void launch_add_vec(const float* a, const float* b, float* out, int n, cudaStream_t s) {
  add_vec_kernel<<<grid_for(n, 256), 256, 0, s>>>(a, b, out, n);
  MDB_LAUNCH_CHECK();
}

// ------------------------------------------------------------------ sub-pixel upsample-conv weights
__global__ void upconv_weights_kernel(const float* __restrict__ w, float* __restrict__ w8, long long pairs) {
  const long long total = pairs * 64;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int e = (int)(i & 7), par = (int)((i >> 3) & 7);
    const long long oc = i >> 6;  // (co, ci) pair
    const int ez = e >> 2, ey = (e >> 1) & 1, ex = e & 1;
    const int pz = par >> 2, py = (par >> 1) & 1, px = par & 1;
    // original taps folded into effective tap (parity q, e): q=0: e0 <- {0}, e1 <- {1,2}; q=1: e0 <- {0,1}, e1 <- {2}
    auto lo = [](int q, int t) { return q == 0 ? (t == 0 ? 0 : 1) : (t == 0 ? 0 : 2); };
    auto hi = [](int q, int t) { return q == 0 ? (t == 0 ? 0 : 2) : (t == 0 ? 1 : 2); };
    float acc = 0.f;
    for (int dz = lo(pz, ez); dz <= hi(pz, ez); ++dz)
      for (int dy = lo(py, ey); dy <= hi(py, ey); ++dy)
        for (int dx = lo(px, ex); dx <= hi(px, ex); ++dx) acc += w[oc * 27 + (dz * 3 + dy) * 3 + dx];
    w8[((long long)par * pairs + oc) * 8 + e] = acc;
  }
}
void launch_upconv_weights(const float* w, float* w8, int Cout, int Cin, cudaStream_t s) {
  const long long pairs = (long long)Cout * Cin;
  upconv_weights_kernel<<<grid_for(pairs * 64, 256), 256, 0, s>>>(w, w8, pairs);
  MDB_LAUNCH_CHECK();
}

// ------------------------------------------------------------------ ancestral sampling update
// Same operation order as the reference's eager fp32 ops (no FMA contraction) so that, given identical eps and
// noise, x and x_mean are bit-identical: score = -eps/std; x_mean = (x + beta*score)/sqrt(1-beta);
// x = x_mean + sqrt(beta)*z; both multiplied by grid_mask (sampling.py:222-230, 476-478).
__global__ void sampler_update_kernel(SamplerUpdateArgs a, int B, float sqrt_1m_beta, float sqrt_beta, float stdv) {
  const long long per = a.V * a.C;
  const long long total = per * B;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long v = i % a.V;
    const float m = __ldg(a.mask + v);
    const float score = __fdiv_rn(-a.eps[i], stdv);
    const float xm = __fdiv_rn(__fadd_rn(a.x[i], __fmul_rn(a.beta, score)), sqrt_1m_beta);
    float z;
    if (a.noise) {
      z = a.noise[i];
    } else {
      curandStatePhilox4_32_10_t st;
      curand_init(a.seed, (unsigned long long)i, a.offset, &st);
      z = curand_normal(&st);
    }
    const float xn = __fadd_rn(xm, __fmul_rn(sqrt_beta, z));
    float xo = __fmul_rn(xn, m), xmo = __fmul_rn(xm, m);
    if (a.cond_partial) {
      const long long bc = i / a.V;
      const int ch = (int)(bc % a.C);
      if (ch == a.cond_channel) {
        const long long b = bc / a.C;
        const float pm = __ldg(a.cond_pmask + b * a.cond_pmask_bs + v);
        const float pv = __ldg(a.cond_partial + b * a.cond_partial_bs + v);
        const float keep = __fsub_rn(1.f, pm);
        const float x1 = __fmul_rn(__fadd_rn(__fmul_rn(xo, keep), __fmul_rn(pv, pm)), m);
        float z2;
        if (a.cond_noise) {
          z2 = a.cond_noise[b * a.V + v];
        } else {
          curandStatePhilox4_32_10_t st;
          curand_init(a.seed, (unsigned long long)i, a.offset + 2, &st);
          z2 = curand_normal(&st);
        }
        const float sampled = __fadd_rn(__fmul_rn(a.cond_coef, x1), __fmul_rn(a.cond_std, z2));
        xo = __fmul_rn(__fadd_rn(__fmul_rn(x1, keep), __fmul_rn(sampled, pm)), m);
        xmo = xo;
      }
    }
    a.x[i] = xo;
    a.x_mean[i] = xmo;
  }
}
void launch_sampler_update(const SamplerUpdateArgs& a, int B, cudaStream_t s) {
  const float one_m = 1.f - a.beta;
  const float sq1m = sqrtf(one_m), sqb = sqrtf(a.beta);
  sampler_update_kernel<<<grid_for(a.V * a.C * B, 256), 256, 0, s>>>(a, B, sq1m, sqb, a.stdv);
  MDB_LAUNCH_CHECK();
}

__global__ void mask_mul_kernel(float* x, const float* mask, long long V, long long total) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x)
    x[i] *= __ldg(mask + (i % V));
}
void launch_mask_mul(float* x, const float* mask, long long V, int C, int B, cudaStream_t s) {
  const long long total = V * C * B;
  mask_mul_kernel<<<grid_for(total, 256), 256, 0, s>>>(x, mask, V, total);
  MDB_LAUNCH_CHECK();
}

}  // namespace mdb

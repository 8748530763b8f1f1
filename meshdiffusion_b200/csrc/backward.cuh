// Bandwidth-bound kernels of the score-network backward pass (what torch autograd runs for the reference's
// loss.backward(), lib/diffusion/losses.py:104-139): GroupNorm(+SiLU, +dropout) backward, bias / time-embedding
// column sums, the data movement of Down/Upsample backward, attention softmax backward and the time-embedding MLP.
// Every reduction is staged (per-thread -> per-block partial -> fixed-order final sum): gradients are bitwise
// reproducible run to run.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>

namespace mdb {

// total block budget of the staged reductions: grid = (ceil(kBwdTargetBlocks / B), B). Partial buffers hold
// kBwdPartRows(B) rows of C (or 2C) floats.
constexpr int kBwdTargetBlocks = 592;
inline int kBwdPartRows(int B) { return kBwdTargetBlocks + B; }

// GroupNorm(32, eps 1e-6) [+SiLU] [+dropout] backward over the channel concatenation of up to two sources.
//   forward:  y = gamma*xhat + beta, a = drop(act(y));   given da = dL/da  [B][V][C] dense
//   pass 1 (reduce): S1[b][c] = sum_v dy, S2[b][c] = sum_v dy*xhat           (dy = da * act'(y) * drop)
//   pass 2 (apply):  dx = rstd*(gamma*dy - mean_g(gamma*dy) - xhat*mean_g(gamma*dy*xhat)) + add0 + add1
//   Pass 1 stores dy over da, so the activation derivative and the dropout hash are evaluated once per element.
struct GnBwdArgs {
  const void* x0; int C0; long long ld0;   // forward input (raw), first source
  const void* x1; int C1; long long ld1;   // second (concatenated) source or null
  const long long* stats0; const long long* stats1;  // forward statistics of the sources ([B][Ci][kStatWords], gn_stats.cuh)
  const float* gamma; const float* beta;
  const void* da;          // [B][V][C] dense, activation dtype; OVERWRITTEN with dy by pass 1 (pass 2 reads dy from it)
  long long voxels; int silu; int groups; float eps;
  // dropout that followed the activation in the forward pass (keep iff hash16(seed, element) >= drop_thresh)
  int drop_thresh; float drop_scale; unsigned long long seed;
  // pass 1 output / pass 2 input
  float* part;             // [gx][B][C][2] block partials (scratch)
  float* sums;             // [B][C][2]
  float* dgamma; float* dbeta; int accumulate;  // parameter gradients (+= when accumulate)
  // pass 2
  void* dx;                // [B][V][C] dense
  const void* add0; long long add0_ld;
  const void* add1; long long add1_ld;
  // optional by-product of pass 2: cs_per[b][c] = sum_v dx[b][v][c] (cs_part: [rows][C] block partials)
  float* cs_part; float* cs_per;
  // 1: x0, x1, da, dx, add0, add1 are split-bf16 tensors ((hi, lo) rows, gemm_host.h::kBF16X3; pitches stay logical)
  int x3;
};
void launch_gn_bwd_reduce(const GnBwdArgs& a, int B, cudaStream_t s);  // part -> sums -> dgamma/dbeta
void launch_gn_bwd_apply(const GnBwdArgs& a, int B, cudaStream_t s);

// Fused variant: the data-gradient GEMM that produces `da` applies dy = da*drop*act'(y) in its epilogue (gemm_tc.cuh,
// GNB) and leaves per-tile column partials; pass 1 above is then replaced by these two small kernels.
// consts[b][c] = {0.5*rstd*gamma, 0.5*(beta - mean*rstd*gamma), rstd, -mean*rstd}
void launch_gn_consts(const GnBwdArgs& a, float* consts4, int B, cudaStream_t s);
// sums[b][c][2] = sum over the T tiles of sample b of part[((b/bb*T + t)*bb + b%bb)][c][2]; then dgamma / dbeta
void launch_gnb_tile_reduce(const GnBwdArgs& a, const float* tile_part, int T, int bb, int B, cudaStream_t s);

// colsum: per[b][c] = sum_v t[b][v][c]; total[c] (+)= sum_b per[b][c]. `per` (nullable) is written with row pitch
// per_ld; up to three `total` outputs receive the same values (conv bias + folded shortcut bias, stem biases).
struct ColsumArgs {
  const void* t; long long ld; int C; long long voxels;
  float* part;                // [gx][B][C] scratch
  float* per; long long per_ld;
  float* total0; float* total1; float* total2; int accumulate;
  const float* from_per; long long from_ld;  // per-sample sums already computed by the producing kernel ([B][from_ld])
  int x3;                     // t is a split-bf16 tensor ((hi, lo) rows of logical pitch ld)
};
void launch_colsum(const ColsumArgs& a, int B, cudaStream_t s);

// Downsample backward helper: z[b][2i+1 (each axis)][c] = dy[b][i][c], zero elsewhere (z has twice the extents).
// Moves whole rows: a split-bf16 tensor is passed as 2C bf16 channels.
void launch_zero_stuff2x(const void* dy, void* z, int B, int R, int C, cudaStream_t s);
// Upsample backward: dx[b][i][c] = sum over the 2x2x2 block of d_up (R = extents of dx). x3: split-bf16 rows.
void launch_downsum2x(const void* dup, void* dx, int B, int R, int C, int x3, cudaStream_t s);
// out[v][c] = sum_b t[b][v][c]  (bf16, VC = voxels * C; x3: split-bf16 rows of C channels)
void launch_batch_sum(const void* t, void* out, int B, long long VC, int C, int x3, cudaStream_t s);
// out[c] (+)= sum_{b,v} t[b][c][v]  (fp32 NCDHW, e.g. the head bias gradient)
void launch_rowsum_nc(const float* t, float* out, int B, int C, long long V, int accumulate, cudaStream_t s);

// Attention softmax backward, in place: row r holds dP (fp32, L values); P holds the probabilities written by the
// forward softmax (bf16 at the start of rows of L fp32 slots). Writes dS = P*(dP - sum(P*dP)) as bf16 at the start of
// each dP row (same convention as the forward). x3: P and dS as [L hi | L lo] bf16 in the row's L fp32 slots.
void launch_softmax_bwd_rows(const float* P, float* dP, long long rows, int L, int x3, cudaStream_t s);

// dW[n][k] (+)= sum_b dy[b][n] x[b][k];  db[n] (+)= sum_b dy[b][n]      (fp32, small)
void launch_outer_sum(const float* dy, long long dy_ld, const float* x, long long x_ld, float* dW, float* db, int B, int N, int K,
                      int accumulate, cudaStream_t s);
// dx[b][k] = sum_n dy[b][n] W[n][k]
void launch_dense_bwd_input(const float* dy, long long dy_ld, const float* W, float* dx, int B, int N, int K, cudaStream_t s);
// time-embedding MLP backward (recomputes the forward from labels): given d(act(temb)) [B][4nf] produces
// dt2, h1 [B][4nf] and dt1 [B][4nf], emb [B][nf] for the outer-product weight gradients.
void launch_temb_bwd(const float* labels, const float* w0, const float* b0, const float* w1, const float* b1, const float* dact,
                     float* dt2, float* h1, float* dt1, float* emb, int B, int nf, cudaStream_t s);

// 16-bit dropout hash shared by the forward GroupNorm-apply kernel and its backward
__device__ __forceinline__ unsigned long long drop_hash64(unsigned long long seed, unsigned long long idx) {
  unsigned long long z = idx + seed * 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

}  // namespace mdb

// Bandwidth-bound kernels around the tcgen05 contractions: GroupNorm finalize/apply (+SiLU), nearest 2x upsample,
// stem im2col, attention softmax / V transpose, time-embedding MLP, ancestral-sampling update.
// All of these are HBM-roofline kernels: 16-byte vector accesses, grid-stride loops sized to the SM count.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>

namespace mdb {

struct GnFinalizeArgs {
  const long long* stats0; int C0;   // [B][C0][kStatWords] split fixed-point (sum, sumsq) records (gn_stats.cuh)
  const long long* stats1; int C1;   // optional second (concatenated) source
  const float* gamma; const float* beta;
  float* scale; float* shift;     // [B][C0+C1]
  int groups; float eps; double count_per_channel;  // voxels per channel
};
void launch_gn_finalize(const GnFinalizeArgs& a, int B, cudaStream_t s);

// y[b][v][c] = act(x[b][v][c] * scale[b][c] + shift[b][c]) over the channel concatenation of up to 2 sources.
struct NormActArgs {
  const void* x0; int C0; long long ld0;
  const void* x1; int C1; long long ld1;
  const float* scale; const float* shift;  // [B][C0+C1] (only when stats0 == nullptr: precomputed by gn_finalize)
  void* y;                                 // [B][V][C0+C1] dense
  long long voxels; int silu; int tf32;  // tf32: storage mode 0 = bf16, 1 = fp32 (tf32 operands), 2 = split bf16 (hi | lo rows)
  // fused GroupNorm finalize: per-channel (sum, sumsq) records of the two sources (gn_stats.cuh), affine parameters
  const long long* stats0; const long long* stats1;
  const float* gamma; const float* beta;
  int groups; float eps;
  // training: nn.Dropout after the activation (layers.py:661,682): keep iff hash16(seed, element) >= drop_thresh
  int drop_thresh; float drop_scale; unsigned long long seed;
};
void launch_norm_act(const NormActArgs& a, int B, cudaStream_t s);

void launch_upsample2x(const void* x, void* y, int B, int Z, int Y, int X, int C, int tf32, cudaStream_t s);

// x fp32 NCDHW [B][Cin][R^3] -> A[b][voxel][Kpad], column = cin*k^3 + tap (tap = (kd*k+kh)*k+kw), zero padded.
void launch_im2col(const float* x, void* a, int B, int Cin, int R, int ksize, int Kpad, int tf32, cudaStream_t s);

// in-place row softmax: rows of L fp32 logits (row stride L floats); writes probabilities in the activation dtype
// at the start of each row (bf16 rows keep the fp32 row pitch).
void launch_softmax_rows(float* s, long long rows, int L, int tf32, cudaStream_t st);

// out[b][c][v] = in[b][v][c0 + c]
void launch_transpose_vc(const void* in, long long ld_in, int c0, void* out, int B, int V, int C, int tf32,
                         cudaStream_t s, long long ld_out = 0);
// the same for bf16 operand matrices of logical pitch ld; x3: (hi, lo) rows [ld hi | ld lo] -> [V hi | V lo] rows
void launch_transpose_vc_rows(const void* in, long long ld, int c0, void* out, int B, int V, int C, int x3, cudaStream_t s);

// temb path (ddpm_res64.py:132-136 + layers.py:542-556,680): act(temb)[B][4nf]
void launch_temb(const float* labels, const float* w0, const float* b0, const float* w1, const float* b1, float* out,
                 int B, int nf, cudaStream_t s);
// out[b][n] = W[n][:] . x[b][:] + bias[n]   (all Dense_0 projections at once)
void launch_dense(const float* x, const float* w, const float* bias, float* out, int B, int K, int N, cudaStream_t s);

// Head convolution, second phase: out[b][co][v] = bias[co] + sum_taps P[b][v + off(tap)][tap*Cout + co] (zero outside the
// grid). P holds the per-tap projections of the normalised activations ([B][V][ldp], activation dtype or fp32).
void launch_tap_shift_sum(const void* P, long long ldp, int p_fp32, const float* bias, float* out, int B, int R, int k,
                          int Cout, cudaStream_t s);

// Split-K reduction + the GEMM epilogue terms: out[b][v][n] = sum_s partial[s][b][v][n] + bias[n] + rowbias[b][n] +
// res[b][v][n], stored in the activation dtype, with the per-(sample, channel) GroupNorm statistics.
struct SplitReduceArgs {
  const float* partial; long long split_stride; int splits;
  const float* bias; const float* rowbias; long long rowbias_ld;
  const void* res; long long res_batch_stride;  // same [V][N] layout as out (activation dtype)
  void* out; long long* stats; long long voxels; int N; int tf32;
};
void launch_split_reduce(const SplitReduceArgs& a, int B, cudaStream_t s);

void launch_add_vec(const float* a, const float* b, float* out, int n, cudaStream_t s);

// Sub-pixel form of Upsample(nearest x2) + conv3^3 (layers.py:611-623): w OIDHW [Cout][Cin][3][3][3] -> w8
// [8 parities (pz,py,px)][Cout][Cin][2][2][2] with, per axis, parity 0: {W0, W1+W2}, parity 1: {W0+W1, W2}.
void launch_upconv_weights(const float* w, float* w8, int Cout, int Cin, cudaStream_t s);

// Ancestral-sampling predictor update fused with the score scaling and both mask multiplies
// (sampling.py:222-230,476-478; models/utils.py:191-198). All fp32, NCDHW [B][4][V]; mask [V].
struct SamplerUpdateArgs {
  const float* eps;    // network output
  float* x;            // in/out state
  float* x_mean;       // out
  const float* noise;  // z ~ N(0,1) or null (then Philox below)
  const float* mask;   // [V]
  float beta, stdv;    // beta_t, sqrt(1-alpha_bar_t)
  long long V; int C;
  unsigned long long seed, offset;  // Philox stream for in-kernel noise
  // replacement conditioning of pc_sampler's partial branch (sampling.py:453-467), applied to channel cond_channel after
  // the masked predictor update when cond_partial != nullptr:
  //   x_c <- (x_c (1-pm) + partial pm) g;  s = coef x_c + std z';  x_c <- (x_c (1-pm) + s pm) g;  x_mean_c <- x_c
  const float* cond_partial; long long cond_partial_bs;  // channel c of sample 0, sample stride (0 = shared grid)
  const float* cond_pmask; long long cond_pmask_bs;
  int cond_channel;
  float cond_coef, cond_std;     // marginal_prob(x, t_i): exp(log_mean_coeff), sqrt(1 - exp(2 log_mean_coeff))
  const float* cond_noise;       // z' [B][V] or null (then Philox(seed, element, offset + 2))
};
void launch_sampler_update(const SamplerUpdateArgs& a, int B, cudaStream_t s);

void launch_mask_mul(float* x, const float* mask, long long V, int C, int B, cudaStream_t s);

}  // namespace mdb

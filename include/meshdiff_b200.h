/* meshdiff_b200 -- C ABI of the B200-native MeshDiffusion hot path.
 *
 * The reference (lzzcd001/MeshDiffusion) has no FFI on this path: its seam is a set of Python callables
 * (SURVEY.md section 8b). Each entry point below names the reference callable it replaces. All pointers are raw
 * device pointers unless stated otherwise; `stream` is a cudaStream_t passed as void*. Every function returns 0 on
 * success and a non-zero code on failure, with a message available from mdb_last_error(). Nothing here
 * synchronises the stream except where stated, and nothing allocates caller-visible memory.
 */
#ifndef MESHDIFF_B200_H
#define MESHDIFF_B200_H

#ifdef __cplusplus
extern "C" {
#endif

const char* mdb_last_error(void);
int mdb_version(void);

/* ------------------------------------------------------------------------------------------------------------
 * Score network. Replaces DDPMRes64 / DDPMRes128 construction + forward
 * (lib/diffusion/models/ddpm_res64.py:41-199, ddpm_res128.py:43-215) as created by
 * mutils.create_model (lib/diffusion/models/utils.py:88-96).
 */
typedef struct mdb_unet mdb_unet;

typedef struct mdb_unet_config {
  int image_size;          /* config.data.image_size */
  int nf;                  /* config.model.nf */
  int n_levels;            /* len(config.model.ch_mult) */
  int ch_mult[8];          /* config.model.ch_mult */
  int num_res_blocks;      /* config.model.num_res_blocks */
  int level0_blocks;       /* ddpm_res128.py:98 forces 2 at level 0; -1 = num_res_blocks */
  int n_attn;
  int attn_resolutions[4]; /* config.model.attn_resolutions */
  int num_channels;        /* config.data.num_channels */
  int stem_ksize;          /* 3 = ddpm_conv3x3 (res64), 5 = ddpm_conv5x5 (res128) */
  int use_pos_bias;        /* 1: stem adds pos_layer(coords*0) = its bias (ddpm_res64.py:148) */
  int max_batch;
  int precision;           /* 0 = bf16 operands, 1 = tf32 operands, 2 = split bf16 ("bf16x3": every value is a (hi, lo)
                              bf16 pair and every product hi*hi + hi*lo + lo*hi -- fp32-class results, the mode that
                              meets the 1e-3 parity contract); fp32 accumulation in all three */
  int training;            /* 1 = also build the backward plan and keep what it needs; precision 0 (bf16) or 2 (bf16x3:
                              split-bf16 activations, data and weight gradients for fp32-class gradients), not tf32 */
} mdb_unet_config;

int mdb_unet_create(const mdb_unet_config* cfg, mdb_unet** out);
/* Plan only (parameter table, arena size); no GPU needed. forward()/set_param() must not be called on it. */
int mdb_unet_create_dry(const mdb_unet_config* cfg, mdb_unet** out);
void mdb_unet_destroy(mdb_unet* net);

/* Parameter table == the reference state_dict without the DataParallel `module.` prefix
 * (lib/diffusion/utils.py:23-30). Shapes are the reference's (OIDHW conv weights, [in,out] NIN.W, ...). */
int mdb_unet_num_params(mdb_unet* net);
int mdb_unet_param_info(mdb_unet* net, int idx, const char** name, long long* numel, int* ndim, long long* shape8);
/* load_state_dict: copy one tensor in (src on host if src_is_device == 0). */
int mdb_unet_set_param(mdb_unet* net, const char* name, const float* src, long long numel, int src_is_device,
                       void* stream);
/* The same for `count` DEVICE tensors in one call (the training step re-uploads all ~500 master parameters after every
 * optimiser step, losses.py:26-52: one host call instead of 500). */
int mdb_unet_set_params(mdb_unet* net, int count, const char* const* names, const float* const* srcs, const long long* numels,
                        void* stream);
/* state_dict: copy one tensor out; synchronises the stream. */
int mdb_unet_get_param(mdb_unet* net, const char* name, float* dst, long long numel, int dst_is_device, void* stream);
/* Re-derive packed weights / constant stem field after parameters changed; synchronises the stream. */
int mdb_unet_commit(mdb_unet* net, void* stream);
/* score_model(x, labels): x fp32 NCDHW [B][C][R][R][R], labels fp32 [B], out fp32 NCDHW (ddpm_res64.py:126-199). */
int mdb_unet_forward(mdb_unet* net, const float* x, const float* labels, float* out, int batch, void* stream);
int mdb_unet_info(mdb_unet* net, double* flops_per_sample, long long* arena_bytes, int* n_gemm_launches, int* n_steps);
/* One profiled forward: per-step device milliseconds. names_buf receives '\n'-separated step names. Synchronises. */
int mdb_unet_profile(mdb_unet* net, const float* x, const float* labels, float* out, int batch, void* stream,
                     char* names_buf, int names_len, float* ms, int max_steps, int* n_steps);

/* ---- training (engines created with cfg.training = 1). Replaces `loss.backward()` through score_model
 * (lib/diffusion/losses.py:104-139 -> torch autograd over ddpm_res64.py:126-199).
 * Dropout of the next forward/backward pair (nn.Dropout(p) after GroupNorm_1+SiLU, layers.py:661,682); p = 0 is
 * model.eval(). The same (p, seed) must be in force for a forward and its backward. */
int mdb_unet_set_dropout(mdb_unet* net, float p, unsigned long long seed);
/* dout = dL/d(out) of the immediately preceding mdb_unet_forward (same x, labels, batch; x and labels must still be
 * alive). grads: ONE flat fp32 buffer of grads_numel = sum of all parameter numels, parameter i at the offset
 * mdb_unet_grad_offset gives (table order); slots of non-trainable tensors (mask, coords, sigmas, pos_layer.weight,
 * whose input is coords*0) are not written. accumulate != 0: grads += (micro-batching, losses.py:111-113). */
int mdb_unet_backward(mdb_unet* net, const float* dout, float* grads, long long grads_numel, int batch, int accumulate,
                      void* stream);
int mdb_unet_grad_offset(mdb_unet* net, const char* name, long long* offset);
/* Data-parallel overlap (replaces the gradient gather of nn.DataParallel, lib/diffusion/models/utils.py:95): the backward
 * plan is a fixed launch list; mdb_unet_grad_ready gives, per parameter, the number of launches after which its gradient
 * is final (0 = never written). mdb_unet_backward_marked is mdb_unet_backward that additionally records the caller's CUDA
 * events (cudaEvent_t as void*) on `stream` once mark_steps[j] launches (ascending) have been enqueued, so the host can
 * all-reduce a finished range of the flat buffer on another stream while the remaining launches run. */
int mdb_unet_grad_ready(mdb_unet* net, const char* name, int* n_launches);
int mdb_unet_backward_marked(mdb_unet* net, const float* dout, float* grads, long long grads_numel, int batch,
                             int accumulate, const int* mark_steps, void* const* mark_events, int n_marks, void* stream);
/* Diagnostics: copies the raw GroupNorm statistics of the last forward to the host (split fixed-point records (sum lo, sum hi,
 * sumsq lo, sumsq hi), per tensor [B][C][4] in plan order); synchronises. count receives the number of int64 values. */
int mdb_unet_debug_stats(mdb_unet* net, long long* host_out, long long capacity, long long* count);
int mdb_unet_train_info(mdb_unet* net, double* bwd_flops_per_sample, int* n_bwd_steps, long long* total_param_numel);
/* One profiled backward (same contract as mdb_unet_profile). */
int mdb_unet_profile_backward(mdb_unet* net, const float* dout, float* grads, int batch, void* stream, char* names_buf,
                              int names_len, float* ms, int max_steps, int* n_steps);

/* Position-weighted 64-bit fingerprints of n fp32 device tensors (ptrs_dev / numels_dev / out_dev are device
 * arrays of n entries). Host plumbing for load_state_dict-style change detection; no reference counterpart. */
int mdb_fingerprint(const void* const* ptrs_dev, const long long* numels_dev, int n, unsigned long long* out_dev,
                    void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Sampler. Replaces AncestralSamplingPredictor.vpsde_update_fn + get_score_fn + the two grid_mask multiplies of
 * pc_sampler (lib/diffusion/sampling.py:222-230, 469-478; lib/diffusion/models/utils.py:191-198).
 * eps = network output, x / x_mean fp32 NCDHW [B][C][V], mask [V]; noise may be NULL (then Philox(seed, offset)).
 */
/* Replacement conditioning of pc_sampler's partial branch (`cond_gen`; lib/diffusion/sampling.py:453-467), fused into the
 * same update kernel. After the masked predictor update, on channel `channel` only (g = grid mask, pm = partial_mask):
 *   x_c <- (x_c (1 - pm) + partial pm) g;   s = mean_coef x_c + std z';   x_c <- (x_c (1 - pm) + s pm) g;   x_mean_c <- x_c
 * with (mean_coef, std) = VPSDE.marginal_prob(., t_i) (sde_lib.py:210-214). partial / partial_mask point at channel
 * `channel` of sample 0 ([V] floats); *_bstride is the element distance to the next sample (0 = one grid shared by the
 * whole batch, the (1,1,R,R,R) tensors evaler.py:181-201 builds). noise: z' [B][V], or NULL for Philox(seed, offset + 2). */
typedef struct mdb_sampler_cond {
  const float* partial;
  long long partial_bstride;
  const float* partial_mask;
  long long mask_bstride;
  int channel;
  float mean_coef, std; /* mdb_sampler_update only (mdb_sampler_run takes per-step tables) */
  const float* noise;
} mdb_sampler_cond;

/* Philox: element e of step i draws its predictor noise from counter block (seed, subsequence e, offset); `offset` counts
 * 32-bit outputs and a normal consumes two, so callers stepping a loop pass offset = 4 * i (mdb_sampler_run does). */
int mdb_sampler_update(const float* eps, float* x, float* x_mean, const float* noise, const float* mask, float beta,
                       float std, long long voxels, int channels, int batch, unsigned long long seed,
                       unsigned long long offset, const mdb_sampler_cond* cond /* nullable */, void* stream);
/* Whole predictor loop of pc_sampler (unconditional branch sampling.py:469-478; partial branch :441-467 when `cond` is
 * given) without host round trips: for i < n_steps: labels[i] -> network -> update [-> replacement conditioning while
 * step0 + i < cond_until, i.e. min(freeze_iters, N - 1)]. labels/betas/stds (and cond_mean_coefs/cond_stds) are HOST
 * arrays of n_steps floats for the global steps step0 .. step0 + n_steps - 1. eps_buf: device scratch [B][C][V];
 * labels_buf: device scratch [B]. Noise is in-kernel Philox at offset 4 * (step0 + i). The call only enqueues work. */
int mdb_sampler_run(mdb_unet* net, float* x, float* x_mean, const float* mask, const float* labels,
                    const float* betas, const float* stds, int n_steps, int batch, unsigned long long seed,
                    float* eps_buf, float* labels_buf, int step0, const mdb_sampler_cond* cond /* nullable */,
                    const float* cond_mean_coefs, const float* cond_stds, int cond_until, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Training-step kernels (optimiser side). Replace get_ddpm_loss_fn's elementwise tail (lib/diffusion/losses.py:69-78),
 * torch.nn.utils.clip_grad_norm_ + torch.optim.Adam.step (losses.py:45-50, 26-35) and
 * ExponentialMovingAverage.update (lib/diffusion/models/ema.py:43-64). Pointer tables / numels are DEVICE arrays of
 * n entries (one per parameter tensor). The multi-tensor passes walk a CHUNK TABLE the host builds once: a device array of
 * n_chunks (tensor index, chunk index) int32 pairs covering every tensor in pieces of mdb_chunk_elems() elements.
 */
/* loss = mean_b[mean_{c,v}((pred-noise)^2 mask[v])] * V / mask_sum -> *loss_out; grad_pred (nullable) = dloss/dpred.
 * scratch: one device double. */
int mdb_ddpm_loss(const float* pred, const float* noise, const float* mask, double mask_sum, float* loss_out,
                  float* grad_pred, double* scratch, int batch, int channels, long long voxels, void* stream);
/* x_t = (sqrt_ac[b] x_0 + sqrt_1mac[b] eps) * mask[v] (losses.py:63-66), fp32 NCDHW [B][C][V]; coefficient arrays [B] on
 * the device; same rounding as the eager torch expression. */
int mdb_ddpm_perturb(const float* x0, const float* noise, const float* mask, const float* sqrt_ac,
                     const float* sqrt_1mac, float* out, int batch, int channels, long long voxels, void* stream);
int mdb_chunk_elems(void);
/* clip_grad_norm_ (losses.py:49): coef = min(1, max_norm / (||g||_2 + 1e-6)) over all tensors -> *coef_out (and the norm
 * in *total_norm_out); the gradients themselves are NOT rescaled (mdb_adam_ema_step applies the coefficient on the fly).
 * scratch: n_chunks device doubles (per-chunk partials, summed in a fixed order: reproducible). */
int mdb_grad_clip_coef(const float* const* grads_dev, const long long* numels_dev, const int* chunks_dev, int n_chunks,
                       float max_norm, float* coef_out, float* total_norm_out, double* scratch, void* stream);
/* g *= *clip_coef (nullable); torch.optim.Adam(lr, beta1, beta2, eps, weight_decay) update number `step` >= 1 (losses.py:26-35);
 * then, when ema_dev != NULL, ExponentialMovingAverage.update: ema -= (1 - ema_decay)(ema - p) (ema.py:43-64). One pass. */
int mdb_adam_ema_step(float* const* params_dev, const float* const* grads_dev, float* const* exp_avg_dev,
                      float* const* exp_avg_sq_dev, float* const* ema_dev, const long long* numels_dev,
                      const int* chunks_dev, int n_chunks, float lr, float beta1, float beta2, float eps,
                      float weight_decay, int step, const float* clip_coef_dev, float ema_decay, void* stream);
/* ExponentialMovingAverage.update on its own (micro-steps that accumulate gradients without an optimiser step). */
int mdb_ema_update(float* const* ema_dev, const float* const* params_dev, const long long* numels_dev,
                   const int* chunks_dev, int n_chunks, float ema_decay, void* stream);

/* Data-parallel training: mean all-reduce of the flat gradient buffer (what mdb_unet_backward filled) over the caller's
 * NCCL communicator (ncclComm_t passed as void*), in place, on `stream`; replaces nn.DataParallel's gradient gather
 * (lib/diffusion/models/utils.py:95). NCCL is taken from the libnccl.so.2 already loaded in the process. The Python
 * host of this repository uses torch.distributed.all_reduce on the same buffer instead (torch owns its communicator). */
int mdb_allreduce_grads(void* nccl_comm, float* grads, long long numel, int world_size, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Operator-level entry points (parity tests call these like the reference's renderutils tests call its ops).
 * Activations are NDHWC in the operand dtype of `precision` (bf16 or fp32).
 */
/* nn.Conv3d k in {1,3,5}, stride 1 (padding k/2) or stride 2 (Downsample: pad-high + VALID, layers.py:626-643).
 * x: [B][Z][Y][X][Cin] (input extents), w: fp32 OIDHW, y: [B][Zo][Yo][Xo][Cout]. Optional: bias [Cout],
 * rowbias [B][Cout], residual (same layout as y), stats [B][Cout][4] int64 = (sum, sum of squares) of the result as
 * split fixed-point pairs, value = w_lo * 2^-24 + w_hi * 2^16 (csrc/gn_stats.cuh: exact, order-independent, cannot
 * overflow), accumulated with integer atomics (must be zeroed by the caller). */
int mdb_conv3d(const void* x, int batch, int cin, int z, int y_, int x_, const float* w, const float* bias, int cout,
               int ksize, int stride, void* out, const float* rowbias, const void* residual, long long* stats,
               int precision, void* stream);
/* GroupNorm(32, eps=1e-6) [+ SiLU] from channel statistics: x [B][V][C], stats [B][C][4] (split fixed point, as above),
 * y [B][V][C]. */
int mdb_groupnorm_act(const void* x, const long long* stats, const float* gamma, const float* beta, void* y, int batch,
                      long long voxels, int channels, int silu, int precision, void* stream);

/* Backward of mdb_conv3d (k = 3 stride 1 | 2, or k = 1) in the training operand modes, precision 0 (bf16) or 2 (bf16x3):
 * what autograd's conv3d backward returns. dy: [B][Zo][Yo][Xo][Cout], x: [B][Z][Y][X][Cin] (NDHWC, operand dtype), w: fp32
 * OIDHW. dy_ld / x_ld: logical row pitches in channels (0 = dense); a channel view is a pointer offset plus a pitch, and in
 * bf16x3 its lo half sits one logical row (ld) behind its hi half. dw (nullable): fp32 OIDHW, += when accumulate != 0.
 * dx (nullable; dense [B][Z][Y][X][Cin], operand dtype): stride 2 is the transposed convolution the training plan runs
 * (dy zero-stuffed to the input extents, then the stride-1 data gradient; needs dense dy and cubic extents).
 * batch_plan >= batch (0 = batch): the operations are planned for batch_plan and launched for batch. splits > 1: the data
 * gradient runs split-K with that factor (fp32 partials + the split reduction); `residual` (nullable, dense like dx) is
 * added to dx. Synchronises. */
int mdb_conv3d_backward(const void* dy, const void* x, const float* w, int batch, int cin, int cout, int z, int y_,
                        int x_, int ksize, int stride, float* dw, void* dx, int precision, long long dy_ld, long long x_ld,
                        int accumulate, int batch_plan, int splits, const void* residual, void* stream);
/* Backward of mdb_groupnorm_act over the channel concatenation of x0 (c0 channels) and x1 (c1, nullable), precision 0 or 2:
 * da = dL/dy [B][V][C] (C = c0 + c1) -> dx [B][V][C], dgamma / dbeta fp32 [C] (+= when accumulate != 0). add0 / add1
 * (nullable, [B][V][C]) are summed into dx. Dropout (p, seed) as in mdb_unet_set_dropout. cs_per (nullable): fp32 [B][C]
 * per-sample column sums of dx. stats0 / stats1: [B][c0|c1][4] split fixed point, as above. `da` is used as scratch
 * (overwritten with the pre-activation gradient). Synchronises. */
int mdb_groupnorm_act_backward(const void* x0, int c0, const void* x1, int c1, const long long* stats0,
                               const long long* stats1, const float* gamma, const float* beta, void* da, const void* add0,
                               const void* add1, void* dx, float* dgamma, float* dbeta, float* cs_per, int batch,
                               long long voxels, int silu, float dropout_p, unsigned long long seed, int precision,
                               int accumulate, void* stream);
/* The fused data-gradient + GroupNorm backward of the training plan: da = the data gradient of a k = 3 (stride 1) or
 * k = 1 convolution with weight w (fp32 OIDHW [cout][C][k^3]) applied to dy ([B][R^3][cout]), consumed in the GEMM
 * epilogue as dL/d(output) of GroupNorm(+SiLU)(+dropout) whose input is the concatenation of x0 (c0) and x1 (c1,
 * nullable); then the per-tile partials are reduced and dx = the GroupNorm input gradient (+ add0 + add1) is applied.
 * Same outputs as mdb_conv3d_backward's dx followed by mdb_groupnorm_act_backward. Fails if the GEMM's tile plan is not
 * the one the partial buffers were sized for. Synchronises. */
int mdb_conv3d_dgrad_gn_backward(const void* dy, const float* w, int batch, int cout, int r, int ksize, const void* x0,
                                 int c0, const void* x1, int c1, const long long* stats0, const long long* stats1,
                                 const float* gamma, const float* beta, const void* add0, const void* add1, void* dx,
                                 float* dgamma, float* dbeta, int silu, float dropout_p, unsigned long long seed,
                                 int precision, void* stream);
/* Bandwidth kernels of the training backward, one launch each (precision 0 = bf16, 2 = bf16x3 (hi, lo) rows). Synchronise.
 * colsum: per [B][per_ld] (nullable) = sum_v t[b][v][c]; total [C] (nullable; += when accumulate) = sum_b per. t has logical
 * pitch ld >= C. from_per (nullable, [B][from_ld] fp32): per-sample sums already computed; only the batch sum runs. */
int mdb_colsum(const void* t, long long ld, int channels, int batch, long long voxels, float* per, long long per_ld,
               float* total, int accumulate, const float* from_per, long long from_ld, int precision, void* stream);
/* Upsample backward: dx [B][R^3][C] = sum over each 2x2x2 block of dup [B][(2R)^3][C]. */
int mdb_downsum2x(const void* dup, void* dx, int batch, int r, int channels, int precision, void* stream);
/* out [V][C] = sum_b t[b][v][c]. */
int mdb_batch_sum(const void* t, void* out, int batch, long long voxels, int channels, int precision, void* stream);
/* Downsample backward helper: z [B][(2R)^3][C] = dy [B][R^3][C] at the odd sites of every axis, zero elsewhere. */
int mdb_zero_stuff2x(const void* dy, void* z, int batch, int r, int channels, int precision, void* stream);
/* Attention softmax backward in place: rows of L fp32 slots; P holds the probabilities as the forward softmax leaves them
 * (bf16 at the start of each row; bf16x3: L hi then L lo), dP the fp32 upstream gradient; dS = P (dP - sum(P dP)) replaces
 * dP in the same format as P. */
int mdb_softmax_bwd_rows(const float* p, float* dp, long long rows, int l, int precision, void* stream);
/* out[b][c][v] = in[b][v][c0 + c] for c < C, in of logical pitch ld; bf16x3: in rows [ld hi | ld lo] -> out rows
 * [V hi | V lo] (the attention backward's operand transposes). */
int mdb_transpose_vc(const void* in, long long ld, int c0, void* out, int batch, int voxels, int channels, int precision,
                     void* stream);
/* im2col of fp32 NCDHW x [B][cin][R^3] -> a [B][R^3][kpad] (column cin*k^3 + tap, zero padded), operand dtype. */
int mdb_im2col(const float* x, void* a, int batch, int cin, int r, int ksize, int kpad, int precision, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Marching tetrahedra. Replaces DMTet.__call__ (nvdiffrec/lib/geometry/dmtet.py:105-163; tables :34-54, map_uv
 * :70-99) for a batch of samples over one static tet grid. Integer outputs (faces, uv_idx, face_to_tet,
 * valid_vert_idx; all int64 like the reference's torch.long) are bit-exact with the reference ordering.
 */
/* tets: HOST int32 [F][4] (the npz `indices`); builds the static sorted edge table on the device. */
int mdb_marching_tets_prepare(const int* tets_host, int n_tets, int n_verts, int max_batch, void** handle);
void mdb_marching_tets_destroy(void* handle);
int mdb_marching_tets_info(void* handle, int* n_edges, int* uv_grid_n);
/* uvs: device fp32 [uv_grid_n^2 * 4][2] */
int mdb_marching_tets_uvs(void* handle, float* uvs, void* stream);
/* Phase 1 (synchronises): sdf device fp32 [B][n_verts]; counts_host[b] = {n_verts_out, n_faces, n_valid_verts}. */
int mdb_marching_tets_count(void* handle, const float* sdf, int batch, int* counts_host, void* stream);
/* Phase 2: pos device fp32 [B][n_verts][3] (pos_batch_stride in floats; 0 = shared). Outputs packed per sample at
 * the given element offsets (device int64 [B]); NULL offsets = samples packed back to back in batch order (the exclusive
 * sums of the phase-1 counts, which the library keeps on the device: no upload needed). */
int mdb_marching_tets_extract(void* handle, const float* pos, long long pos_batch_stride, const float* sdf, int batch,
                              float* verts, long long* faces, long long* uv_idx, long long* face_to_tet,
                              long long* valid_vert_idx, const long long* vert_off, const long long* face_off,
                              const long long* vv_off, void* stream);
/* Backward of the vertex interpolation: what torch autograd computes for DMTet.__call__'s `verts` with respect to `pos_nx3`
 * and `sdf_n` (nvdiffrec/lib/geometry/dmtet.py:125-132 under loss.backward(); every other output is an integer tensor).
 * grad_verts fp32 packed like `verts`; vert_off device int64 [B] (NULL = the offsets of the last phase 1); vertex_ids device
 * uint32 [B][n_edges] = crossing edge -> output row, as copied by mdb_marching_tets_vertex_ids after the forward extract
 * (NULL = the last extract's, still held by the handle). grad_pos fp32 [B][n_verts][3] and grad_sdf fp32 [B][n_verts] are
 * overwritten (either may be NULL). A gather per grid vertex over its incident edges: no atomics, bitwise reproducible. */
int mdb_marching_tets_vertex_ids(void* handle, int batch, unsigned* out, void* stream);
int mdb_marching_tets_backward(void* handle, const float* pos, long long pos_batch_stride, const float* sdf, int batch,
                               const unsigned* vertex_ids, const float* grad_verts, const long long* vert_off,
                               float* grad_pos, float* grad_sdf, void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Mesh post-ops after marching tets (SURVEY 8f-1). Scatter-adds run as 2^-40 fixed-point integer atomics: results are
 * independent of face order (bitwise reproducible).
 */
/* auto_normals (nvdiffrec/lib/render/mesh.py:200-227): v_pos fp32 [Nv][3], faces int64 [F][3] -> v_nrm fp32 [Nv][3]
 * (sum of unnormalised face normals, degenerate -> (0,0,1), safe_normalize), f_nrm fp32 [F][3] (nullable).
 * scratch: device int64 [Nv][3]. */
int mdb_mesh_auto_normals(const float* v_pos, const long long* faces, int n_verts, int n_faces, float* v_nrm, float* f_nrm,
                          long long* scratch, void* stream);
/* compute_tangents (mesh.py:233-277): per-face tangent from positions and texture coordinates, averaged per normal
 * index, Gram-Schmidt against v_nrm. v_tex fp32 [Nt][2]; index arrays int64 [F][3]; v_nrm fp32 [Nn][3] -> v_tng [Nn][3].
 * scratch: device bytes Nn*3*8 + Nn*4. */
int mdb_mesh_compute_tangents(const float* v_pos, const long long* t_pos_idx, const float* v_tex, const long long* t_tex_idx,
                              const float* v_nrm, const long long* t_nrm_idx, int n_nrm, int n_faces, float* v_tng,
                              long long* scratch, void* stream);

#ifdef __cplusplus
}
#endif
#endif

// extern "C" boundary (include/meshdiff_b200.h). Exceptions never cross it: they become error codes + a message.
#include "../../include/meshdiff_b200.h"
#include "unet.h"
#include <cstring>
#include <cmath>
#include <memory>

using namespace mdb;

static thread_local std::string g_err;
namespace mdb { void set_last_error(const std::string& msg) { g_err = msg; } }

#define MDB_API_BEGIN try {
#define MDB_API_END                         \
  }                                         \
  catch (const std::exception& e) {         \
    g_err = e.what();                       \
    return 1;                               \
  }                                         \
  catch (...) {                             \
    g_err = "mdb: unknown error";           \
    return 2;                               \
  }                                         \
  return 0;

struct mdb_unet { UNet* net; };

extern "C" {

const char* mdb_last_error(void) { return g_err.c_str(); }
int mdb_version(void) { return 100; }

static int create_impl(const mdb_unet_config* c, mdb_unet** out, bool dry) {
  MDB_API_BEGIN
  if (!c || !out) throw std::runtime_error("mdb: null argument");
  UNetConfig u;
  u.image_size = c->image_size; u.nf = c->nf; u.n_levels = c->n_levels;
  for (int i = 0; i < 8; ++i) u.ch_mult[i] = c->ch_mult[i];
  u.num_res_blocks = c->num_res_blocks; u.level0_blocks = c->level0_blocks;
  u.n_attn = c->n_attn;
  for (int i = 0; i < 4; ++i) u.attn_resolutions[i] = c->attn_resolutions[i];
  u.num_channels = c->num_channels; u.stem_ksize = c->stem_ksize; u.use_pos_bias = c->use_pos_bias;
  u.max_batch = c->max_batch; u.precision = c->precision; u.training = c->training;
  auto* h = new mdb_unet;
  h->net = nullptr;
  try { h->net = new UNet(u, dry); } catch (...) { delete h; throw; }
  *out = h;
  MDB_API_END
}

int mdb_unet_create(const mdb_unet_config* c, mdb_unet** out) { return create_impl(c, out, false); }
int mdb_unet_create_dry(const mdb_unet_config* c, mdb_unet** out) { return create_impl(c, out, true); }

void mdb_unet_destroy(mdb_unet* n) {
  if (!n) return;
  delete n->net;
  delete n;
}

int mdb_unet_num_params(mdb_unet* n) { return n ? (int)n->net->params().size() : -1; }

int mdb_unet_param_info(mdb_unet* n, int idx, const char** name, long long* numel, int* ndim, long long* shape8) {
  MDB_API_BEGIN
  const auto& ps = n->net->params();
  if (idx < 0 || idx >= (int)ps.size()) throw std::runtime_error("mdb: parameter index out of range");
  if (name) *name = ps[idx].name.c_str();
  if (numel) *numel = ps[idx].numel;
  if (ndim) *ndim = (int)ps[idx].shape.size();
  if (shape8) for (size_t i = 0; i < ps[idx].shape.size() && i < 8; ++i) shape8[i] = ps[idx].shape[i];
  MDB_API_END
}

int mdb_unet_set_param(mdb_unet* n, const char* name, const float* src, long long numel, int dev, void* stream) {
  MDB_API_BEGIN
  n->net->set_param(name, src, numel, dev != 0, (cudaStream_t)stream);
  MDB_API_END
}

int mdb_unet_set_params(mdb_unet* n, int count, const char* const* names, const float* const* srcs, const long long* numels,
                        void* stream) {
  MDB_API_BEGIN
  for (int i = 0; i < count; ++i) n->net->set_param(names[i], srcs[i], numels[i], true, (cudaStream_t)stream);
  MDB_API_END
}

int mdb_unet_get_param(mdb_unet* n, const char* name, float* dst, long long numel, int dev, void* stream) {
  MDB_API_BEGIN
  n->net->get_param(name, dst, numel, dev != 0, (cudaStream_t)stream);
  MDB_API_END
}

int mdb_unet_commit(mdb_unet* n, void* stream) {
  MDB_API_BEGIN
  n->net->commit((cudaStream_t)stream);
  MDB_API_END
}

int mdb_unet_forward(mdb_unet* n, const float* x, const float* labels, float* out, int B, void* stream) {
  MDB_API_BEGIN
  n->net->forward(x, labels, out, B, (cudaStream_t)stream);
  MDB_API_END
}

int mdb_unet_info(mdb_unet* n, double* flops, long long* arena, int* ngemm, int* nsteps) {
  MDB_API_BEGIN
  if (flops) *flops = n->net->flops_per_sample();
  if (arena) *arena = (long long)n->net->arena_bytes();
  if (ngemm) *ngemm = n->net->num_gemm_launches();
  if (nsteps) *nsteps = n->net->num_steps();
  MDB_API_END
}

int mdb_unet_profile(mdb_unet* n, const float* x, const float* labels, float* out, int B, void* stream, char* names,
                     int names_len, float* ms, int max_steps, int* nsteps) {
  MDB_API_BEGIN
  auto r = n->net->profile(x, labels, out, B, (cudaStream_t)stream);
  std::string all;
  int k = 0;
  for (auto& p : r) {
    if (k >= max_steps) break;
    all += p.first; all += "\n";
    ms[k++] = p.second;
  }
  if ((int)all.size() + 1 > names_len) throw std::runtime_error("mdb: names buffer too small");
  std::memcpy(names, all.c_str(), all.size() + 1);
  if (nsteps) *nsteps = k;
  MDB_API_END
}

int mdb_unet_set_dropout(mdb_unet* n, float p, unsigned long long seed) {
  MDB_API_BEGIN
  n->net->set_dropout(p, seed);
  MDB_API_END
}

int mdb_unet_backward(mdb_unet* n, const float* dout, float* grads, long long grads_numel, int B, int accumulate, void* stream) {
  MDB_API_BEGIN
  if (grads_numel != n->net->total_param_numel()) throw std::runtime_error("mdb: gradient buffer has the wrong size");
  n->net->backward(dout, grads, B, accumulate != 0, (cudaStream_t)stream);
  MDB_API_END
}

int mdb_unet_backward_marked(mdb_unet* n, const float* dout, float* grads, long long grads_numel, int B, int accumulate,
                             const int* mark_steps, void* const* mark_events, int n_marks, void* stream) {
  MDB_API_BEGIN
  if (grads_numel != n->net->total_param_numel()) throw std::runtime_error("mdb: gradient buffer has the wrong size");
  if (n_marks > 0 && (!mark_steps || !mark_events)) throw std::runtime_error("mdb: null mark arrays");
  n->net->backward(dout, grads, B, accumulate != 0, (cudaStream_t)stream, mark_steps, mark_events, n_marks);
  MDB_API_END
}

int mdb_unet_grad_ready(mdb_unet* n, const char* name, int* step) {
  MDB_API_BEGIN
  *step = n->net->grad_ready_step(name);
  MDB_API_END
}

int mdb_unet_grad_offset(mdb_unet* n, const char* name, long long* off) {
  MDB_API_BEGIN
  *off = n->net->grad_offset(name);
  MDB_API_END
}

int mdb_unet_debug_stats(mdb_unet* n, long long* host_out, long long capacity, long long* count) {
  MDB_API_BEGIN
  const long long c = (long long)n->net->stats_count();
  if (count) *count = c;
  if (host_out) {
    if (capacity < c) throw std::runtime_error("mdb: stats buffer too small");
    MDB_CUDA_CHECK(cudaMemcpy(host_out, n->net->stats_ptr(), (size_t)c * sizeof(long long), cudaMemcpyDeviceToHost));
  }
  MDB_API_END
}

int mdb_unet_train_info(mdb_unet* n, double* bwd_flops, int* nsteps, long long* numel) {
  MDB_API_BEGIN
  if (bwd_flops) *bwd_flops = n->net->bwd_flops_per_sample();
  if (nsteps) *nsteps = n->net->num_bwd_steps();
  if (numel) *numel = n->net->total_param_numel();
  MDB_API_END
}

int mdb_unet_profile_backward(mdb_unet* n, const float* dout, float* grads, int B, void* stream, char* names, int names_len,
                              float* ms, int max_steps, int* nsteps) {
  MDB_API_BEGIN
  auto r = n->net->profile_backward(dout, grads, B, (cudaStream_t)stream);
  std::string all;
  int k = 0;
  for (auto& p : r) {
    if (k >= max_steps) break;
    all += p.first; all += "\n";
    ms[k++] = p.second;
  }
  if ((int)all.size() + 1 > names_len) throw std::runtime_error("mdb: names buffer too small");
  std::memcpy(names, all.c_str(), all.size() + 1);
  if (nsteps) *nsteps = k;
  MDB_API_END
}

static void set_cond(SamplerUpdateArgs& a, const mdb_sampler_cond* c, float coef, float stdv) {
  if (!c || !c->partial) return;
  if (!c->partial_mask) throw std::runtime_error("mdb: conditional sampling needs partial_mask");
  if (c->channel < 0 || c->channel >= a.C) throw std::runtime_error("mdb: partial_channel out of range");
  a.cond_partial = c->partial; a.cond_partial_bs = c->partial_bstride;
  a.cond_pmask = c->partial_mask; a.cond_pmask_bs = c->mask_bstride;
  a.cond_channel = c->channel; a.cond_coef = coef; a.cond_std = stdv; a.cond_noise = c->noise;
}

int mdb_sampler_update(const float* eps, float* x, float* x_mean, const float* noise, const float* mask, float beta,
                       float stdv, long long V, int C, int B, unsigned long long seed, unsigned long long offset,
                       const mdb_sampler_cond* cond, void* stream) {
  MDB_API_BEGIN
  SamplerUpdateArgs a{};
  a.eps = eps; a.x = x; a.x_mean = x_mean; a.noise = noise; a.mask = mask; a.beta = beta; a.stdv = stdv;
  a.V = V; a.C = C; a.seed = seed; a.offset = offset;
  if (cond) set_cond(a, cond, cond->mean_coef, cond->std);
  launch_sampler_update(a, B, (cudaStream_t)stream);
  MDB_API_END
}

// Order-independent 64-bit fingerprint of fp32 tensors (position-weighted sum of the raw words, integer atomics).
// The Python shell uses it to notice parameter edits that bypass autograd's version counters (`p.data[...] = ...`,
// which is how the reference's trainer writes the grid mask and how its EMA copies weights).
__global__ void fingerprint_kernel(const unsigned int* const* ptrs, const long long* numels, unsigned long long* out) {
  const int t = blockIdx.y;
  const unsigned int* p = ptrs[t];
  const long long n = numels[t];
  unsigned long long h = 0;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    h += (unsigned long long)p[i] * (0x9E3779B97F4A7C15ull * (unsigned long long)(i + 1) | 1ull);
  for (int o = 16; o; o >>= 1) h += __shfl_xor_sync(0xffffffffu, h, o);
  if ((threadIdx.x & 31) == 0 && h) atomicAdd(out + t, h);
}

int mdb_fingerprint(const void* const* ptrs_dev, const long long* numels_dev, int n, unsigned long long* out_dev, void* stream) {
  MDB_API_BEGIN
  cudaStream_t s = (cudaStream_t)stream;
  MDB_CUDA_CHECK(cudaMemsetAsync(out_dev, 0, (size_t)n * 8, s));
  fingerprint_kernel<<<dim3(64, n), 256, 0, s>>>(reinterpret_cast<const unsigned int* const*>(ptrs_dev), numels_dev, out_dev);
  MDB_CUDA_CHECK(cudaGetLastError());
  MDB_API_END
}

__global__ void fill_kernel(float* p, float v, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

int mdb_sampler_run(mdb_unet* n, float* x, float* x_mean, const float* mask, const float* labels, const float* betas,
                    const float* stds, int n_steps, int B, unsigned long long seed, float* eps_buf, float* labels_buf,
                    int step0, const mdb_sampler_cond* cond, const float* cond_mean_coefs, const float* cond_stds,
                    int cond_until, void* stream) {
  MDB_API_BEGIN
  cudaStream_t s = (cudaStream_t)stream;
  const UNetConfig& c = n->net->cfg();
  const long long V = (long long)c.image_size * c.image_size * c.image_size;
  if (cond && cond->partial && (!cond_mean_coefs || !cond_stds)) throw std::runtime_error("mdb: conditional run needs the marginal_prob tables");
  if (cond && cond->noise) throw std::runtime_error("mdb: mdb_sampler_run draws its noise in-kernel (cond->noise must be NULL)");
  for (int i = 0; i < n_steps; ++i) {
    fill_kernel<<<(B + 127) / 128, 128, 0, s>>>(labels_buf, labels[i], B);
    n->net->forward(x, labels_buf, eps_buf, B, s, /*allow_graph=*/true);
    SamplerUpdateArgs a{};
    a.eps = eps_buf; a.x = x; a.x_mean = x_mean; a.noise = nullptr; a.mask = mask; a.beta = betas[i]; a.stdv = stds[i];
    // curand_normal consumes two 32-bit Philox outputs and `offset` counts single outputs: 4*i gives every step its own
    // 128-bit counter block, so the noise of consecutive steps is independent
    a.V = V; a.C = c.num_channels; a.seed = seed; a.offset = 4ull * (unsigned long long)(step0 + i);
    if (cond && step0 + i < cond_until) set_cond(a, cond, cond_mean_coefs[i], cond_stds[i]);
    launch_sampler_update(a, B, s);
  }
  MDB_API_END
}

int mdb_conv3d(const void* x, int B, int cin, int z, int y_, int x_, const float* w, const float* bias, int cout,
               int ksize, int stride, void* out, const float* rowbias, const void* residual, long long* stats,
               int precision, void* stream) {
  MDB_API_BEGIN
  cudaStream_t s = (cudaStream_t)stream;
  const Precision pr = precision_from_int(precision);
  const int xo = x_ / stride, yo = y_ / stride, zo = z / stride;
  GemmOp g;
  g.set_output(pr, xo, yo, zo, B, cout, out, cout, false);
  Act a; a.ptr = const_cast<void*>(x); a.C = cin; a.X = x_; a.Y = y_; a.Z = z; a.B = B;
  if (ksize == 1) g.add_pointwise({a}, w, false);
  else g.add_conv({a}, w, ksize, stride);
  if (bias) g.set_bias(bias);
  if (rowbias) g.set_rowbias(rowbias, cout);
  if (residual) g.set_residual(residual, cout, (long long)xo * yo * zo * cout, false);
  if (stats) g.set_stats(stats);
  g.finalize(s, true);
  g.launch(s);
  MDB_CUDA_CHECK(cudaStreamSynchronize(s));
  MDB_API_END
}

int mdb_groupnorm_act(const void* x, const long long* stats, const float* gamma, const float* beta, void* y, int B,
                      long long V, int C, int silu, int precision, void* stream) {
  MDB_API_BEGIN
  cudaStream_t s = (cudaStream_t)stream;
  NormActArgs na{};
  na.x0 = x; na.C0 = C; na.ld0 = C; na.x1 = nullptr; na.C1 = 0; na.ld1 = 0; na.scale = nullptr; na.shift = nullptr;
  na.y = y; na.voxels = V; na.silu = silu; na.tf32 = (int)precision_from_int(precision);
  na.stats0 = stats; na.stats1 = nullptr; na.gamma = gamma; na.beta = beta; na.groups = 32; na.eps = 1e-6f;
  launch_norm_act(na, B, s);
  MDB_CUDA_CHECK(cudaStreamSynchronize(s));
  MDB_API_END
}

// Device scratch of the operator entry points, freed on every exit path.
struct DevBuf {
  void* p = nullptr;
  explicit DevBuf(size_t bytes) { MDB_CUDA_CHECK(cudaMalloc(&p, bytes ? bytes : 16)); }
  ~DevBuf() { if (p) cudaFree(p); }
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  float* f() const { return static_cast<float*>(p); }
};

static Precision train_precision(int v) {
  const Precision p = precision_from_int(v);
  if (p == kTF32) throw std::runtime_error("mdb: the training kernels take precision 0 (bf16) or 2 (bf16x3)");
  return p;
}

static Act act5(const void* ptr, int C, long long ld, int X, int Y, int Z, int B) {
  Act a;
  a.ptr = const_cast<void*>(ptr); a.C = C; a.ld = ld; a.X = X; a.Y = Y; a.Z = Z; a.B = B;
  return a;
}

int mdb_conv3d_backward(const void* dy, const void* x, const float* w, int B, int cin, int cout, int z, int y_, int x_,
                        int ksize, int stride, float* dw, void* dx, int precision, long long dy_ld, long long x_ld,
                        int accumulate, int B_plan, int splits, const void* residual, void* stream) {
  MDB_API_BEGIN
  cudaStream_t s = (cudaStream_t)stream;
  const Precision pr = train_precision(precision);
  if (B_plan == 0) B_plan = B;
  if (B < 1 || B_plan < B) throw std::runtime_error("mdb: conv3d backward needs 1 <= batch <= batch_plan");
  if (stride != 1 && stride != 2) throw std::runtime_error("mdb: conv3d backward supports stride 1 and 2");
  const int xo = x_ / stride, yo = y_ / stride, zo = z / stride;
  const Act ady = act5(dy, cout, dy_ld, xo, yo, zo, B_plan);
  const Act ax = act5(x, cin, x_ld, x_, y_, z, B_plan);
  if (dw) {
    const int T = ksize * ksize * ksize;
    const WgradPlan pl = plan_wgrad(xo, yo, zo, B_plan, cout, cin, ksize, stride);
    DevBuf scratch(pl.scratch_bytes);
    WgradOut o; o.ptr = dw; o.sm = (long long)cin * T; o.sn = T; o.st = 1;
    WgradOp op;
    op.init(ady, ax, ksize, stride, o, scratch.f(), pr == kBF16X3);
    op.launch(s, B, accumulate != 0);
    MDB_CUDA_CHECK(cudaStreamSynchronize(s));
  }
  if (dx) {
    const long long V = (long long)x_ * y_ * z;
    Act src = ady;
    std::unique_ptr<DevBuf> stuffed;
    if (stride == 2) {
      // the training plan's transposed stride-2 convolution: dY zero-stuffed to the input extents, then the stride-1
      // data gradient with the mirrored kernel (UNet::tape_downsample)
      if (ksize != 3 || (dy_ld && dy_ld != cout) || x_ != y_ || y_ != z)
        throw std::runtime_error("mdb: stride-2 data gradient needs k = 3, dense dy and cubic extents");
      stuffed = std::make_unique<DevBuf>((size_t)B_plan * V * cout * 2 * parts(pr));
      launch_zero_stuff2x(dy, stuffed->p, B, xo, cout * parts(pr), s);
      src = act5(stuffed->p, cout, 0, x_, y_, z, B_plan);
    }
    GemmOp g;
    g.set_output(pr, x_, y_, z, B_plan, cin, dx, cin, false);
    if (ksize == 1) { WSrc ws{w, 1, (long long)cin, 0, cout}; g.add_pointwise_w({src}, &ws); }
    else g.add_conv_dgrad(src, w, cin, ksize);
    if (residual) g.set_residual(residual, cin, V * cin, false);
    std::unique_ptr<DevBuf> partial;
    if (splits > 1) {
      partial = std::make_unique<DevBuf>((size_t)splits * B_plan * V * cin * sizeof(float));
      g.enable_splits(splits, partial->f());
    }
    g.finalize(s, true);
    g.launch(s, B);
    MDB_CUDA_CHECK(cudaStreamSynchronize(s));
  }
  MDB_API_END
}

static GnBwdArgs gn_bwd_args(const void* x0, int c0, const void* x1, int c1, const long long* stats0, const long long* stats1,
                             const float* gamma, const float* beta, const void* add0, const void* add1, void* dx,
                             float* dgamma, float* dbeta, long long V, int silu, float dropout_p, unsigned long long seed,
                             Precision pr) {
  if (dropout_p < 0.f || dropout_p >= 1.f) throw std::runtime_error("mdb: dropout probability out of range");
  GnBwdArgs a{};
  a.x0 = x0; a.C0 = c0; a.ld0 = c0; a.stats0 = stats0;
  a.x1 = x1; a.C1 = x1 ? c1 : 0; a.ld1 = a.C1; a.stats1 = x1 ? stats1 : nullptr;
  a.gamma = gamma; a.beta = beta;
  a.voxels = V; a.silu = silu; a.groups = 32; a.eps = 1e-6f;
  a.drop_thresh = (int)lround((double)dropout_p * 65536.0); a.drop_scale = dropout_p > 0.f ? 1.f / (1.f - dropout_p) : 1.f; a.seed = seed;
  a.dgamma = dgamma; a.dbeta = dbeta;
  const int C = a.C0 + a.C1;
  a.dx = dx; a.add0 = add0; a.add0_ld = C; a.add1 = add1; a.add1_ld = C;
  a.x3 = pr == kBF16X3 ? 1 : 0;
  return a;
}

int mdb_groupnorm_act_backward(const void* x0, int c0, const void* x1, int c1, const long long* stats0, const long long* stats1,
                               const float* gamma, const float* beta, void* da, const void* add0, const void* add1, void* dx,
                               float* dgamma, float* dbeta, float* cs_per, int B, long long V, int silu, float dropout_p,
                               unsigned long long seed, int precision, int accumulate, void* stream) {
  MDB_API_BEGIN
  cudaStream_t s = (cudaStream_t)stream;
  GnBwdArgs a = gn_bwd_args(x0, c0, x1, c1, stats0, stats1, gamma, beta, add0, add1, dx, dgamma, dbeta, V, silu, dropout_p,
                            seed, train_precision(precision));
  const int C = a.C0 + a.C1;
  DevBuf part((size_t)kBwdPartRows(B) * C * 2 * sizeof(float)), sums((size_t)B * C * 2 * sizeof(float));
  std::unique_ptr<DevBuf> cs_part;
  if (cs_per) cs_part = std::make_unique<DevBuf>((size_t)kBwdPartRows(B) * C * sizeof(float));
  a.da = da; a.part = part.f(); a.sums = sums.f(); a.accumulate = accumulate != 0;
  a.cs_part = cs_per ? cs_part->f() : nullptr; a.cs_per = cs_per;
  launch_gn_bwd_reduce(a, B, s);
  launch_gn_bwd_apply(a, B, s);
  MDB_CUDA_CHECK(cudaStreamSynchronize(s));
  MDB_API_END
}

int mdb_conv3d_dgrad_gn_backward(const void* dy, const float* w, int B, int cout, int R, int ksize, const void* x0, int c0,
                                 const void* x1, int c1, const long long* stats0, const long long* stats1, const float* gamma,
                                 const float* beta, const void* add0, const void* add1, void* dx, float* dgamma, float* dbeta,
                                 int silu, float dropout_p, unsigned long long seed, int precision, void* stream) {
  MDB_API_BEGIN
  cudaStream_t s = (cudaStream_t)stream;
  const Precision pr = train_precision(precision);
  if (ksize != 1 && ksize != 3) throw std::runtime_error("mdb: the fused data gradient supports k = 1 and k = 3");
  GnBwdArgs a = gn_bwd_args(x0, c0, x1, c1, stats0, stats1, gamma, beta, add0, add1, dx, dgamma, dbeta, (long long)R * R * R,
                            silu, dropout_p, seed, pr);
  const int C = a.C0 + a.C1;
  // partial buffers sized the way UNet::gn_fuse_attach sizes them
  const Geometry geo = pick_geometry(R, R, R);
  const int T = ((R + geo.bx - 1) / geo.bx) * ((R + geo.by - 1) / geo.by) * ((R + geo.bz - 1) / geo.bz);
  const long long rows = 1LL * T * ((B + geo.bb - 1) / geo.bb) * geo.bb;
  DevBuf consts((size_t)B * C * 4 * sizeof(float)), tile_part((size_t)rows * C * 2 * sizeof(float));
  DevBuf sums((size_t)B * C * 2 * sizeof(float)), da((size_t)B * a.voxels * C * 2 * parts(pr));
  a.da = da.p; a.sums = sums.f();
  GemmOp g;
  g.set_output(pr, R, R, R, B, C, da.p, C, false);
  const Act ady = act5(dy, cout, 0, R, R, R, B);
  if (ksize == 1) { WSrc ws{w, 1, (long long)C, 0, cout}; g.add_pointwise_w({ady}, &ws); }
  else g.add_conv_dgrad(ady, w, C, 3);
  g.set_gn_backward(x0, c0, c0, x1, x1 ? c1 : 0, consts.p, silu, tile_part.f());
  if (g.gnb_tiles_per_batch_tile() != T || g.gnb_bb() != geo.bb || g.gnb_rows() != rows)
    throw std::runtime_error("mdb: GroupNorm-backward tile plan mismatch");
  g.rt_drop_thresh = a.drop_thresh; g.rt_drop_scale = a.drop_scale; g.rt_seed = a.seed;
  g.finalize(s, true);
  launch_gn_consts(a, consts.f(), B, s);
  g.launch(s, B);
  launch_gnb_tile_reduce(a, tile_part.f(), T, geo.bb, B, s);
  launch_gn_bwd_apply(a, B, s);
  MDB_CUDA_CHECK(cudaStreamSynchronize(s));
  MDB_API_END
}

int mdb_colsum(const void* t, long long ld, int C, int B, long long V, float* per, long long per_ld, float* total,
               int accumulate, const float* from_per, long long from_ld, int precision, void* stream) {
  MDB_API_BEGIN
  cudaStream_t s = (cudaStream_t)stream;
  DevBuf part((size_t)kBwdPartRows(B) * C * sizeof(float));
  ColsumArgs a{};
  a.t = t; a.ld = ld ? ld : C; a.C = C; a.voxels = V; a.part = part.f();
  a.per = per; a.per_ld = per_ld; a.total0 = total; a.accumulate = accumulate != 0;
  a.from_per = from_per; a.from_ld = from_ld;
  a.x3 = train_precision(precision) == kBF16X3 ? 1 : 0;
  launch_colsum(a, B, s);
  MDB_CUDA_CHECK(cudaStreamSynchronize(s));
  MDB_API_END
}

int mdb_downsum2x(const void* dup, void* dx, int B, int R, int C, int precision, void* stream) {
  MDB_API_BEGIN
  cudaStream_t s = (cudaStream_t)stream;
  launch_downsum2x(dup, dx, B, R, C, train_precision(precision) == kBF16X3 ? 1 : 0, s);
  MDB_CUDA_CHECK(cudaStreamSynchronize(s));
  MDB_API_END
}

int mdb_batch_sum(const void* t, void* out, int B, long long V, int C, int precision, void* stream) {
  MDB_API_BEGIN
  cudaStream_t s = (cudaStream_t)stream;
  launch_batch_sum(t, out, B, V * C, C, train_precision(precision) == kBF16X3 ? 1 : 0, s);
  MDB_CUDA_CHECK(cudaStreamSynchronize(s));
  MDB_API_END
}

int mdb_zero_stuff2x(const void* dy, void* z, int B, int R, int C, int precision, void* stream) {
  MDB_API_BEGIN
  cudaStream_t s = (cudaStream_t)stream;
  launch_zero_stuff2x(dy, z, B, R, C * parts(train_precision(precision)), s);  // whole (hi, lo) rows
  MDB_CUDA_CHECK(cudaStreamSynchronize(s));
  MDB_API_END
}

int mdb_softmax_bwd_rows(const float* P, float* dP, long long rows, int L, int precision, void* stream) {
  MDB_API_BEGIN
  cudaStream_t s = (cudaStream_t)stream;
  launch_softmax_bwd_rows(P, dP, rows, L, train_precision(precision) == kBF16X3 ? 1 : 0, s);
  MDB_CUDA_CHECK(cudaStreamSynchronize(s));
  MDB_API_END
}

int mdb_transpose_vc(const void* in, long long ld, int c0, void* out, int B, int V, int C, int precision, void* stream) {
  MDB_API_BEGIN
  cudaStream_t s = (cudaStream_t)stream;
  launch_transpose_vc_rows(in, ld, c0, out, B, V, C, train_precision(precision) == kBF16X3 ? 1 : 0, s);
  MDB_CUDA_CHECK(cudaStreamSynchronize(s));
  MDB_API_END
}

int mdb_im2col(const float* x, void* a, int B, int cin, int R, int ksize, int kpad, int precision, void* stream) {
  MDB_API_BEGIN
  cudaStream_t s = (cudaStream_t)stream;
  launch_im2col(x, a, B, cin, R, ksize, kpad, (int)train_precision(precision), s);
  MDB_CUDA_CHECK(cudaStreamSynchronize(s));
  MDB_API_END
}

}  // extern "C"

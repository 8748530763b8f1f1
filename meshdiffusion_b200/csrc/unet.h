// Score-network engine: builds the DDPM 3-D U-Net (reference lib/diffusion/models/ddpm_res64.py:41-199,
// ddpm_res128.py:43-215, layers.py:573-689) as a static plan of tcgen05 GEMM ops + bandwidth kernels over a
// liveness-packed HBM arena, and replays it per denoising step.
#pragma once
#include <functional>
#include <map>
#include <memory>
#include <string>
#include <vector>
#include "gemm_host.h"
#include "wgrad_host.h"
#include "elementwise.cuh"
#include "backward.cuh"

namespace mdb {

struct UNetConfig {
  int image_size = 64;
  int nf = 128;
  int n_levels = 5;
  int ch_mult[8] = {1, 1, 2, 4, 4, 0, 0, 0};
  int num_res_blocks = 3;
  int level0_blocks = -1;  // ddpm_res128.py:98 uses 2 blocks at level 0; -1 = num_res_blocks
  int n_attn = 1;
  int attn_resolutions[4] = {16, 0, 0, 0};
  int num_channels = 4;
  int stem_ksize = 3;   // 3 (res64) or 5 (res128)
  int use_pos_bias = 1; // ddpm_res64.py:148 adds pos_layer(coords*0) == its bias; res128 does not
  int max_batch = 1;
  int precision = 0;    // 0 = bf16 operands, 1 = tf32 operands, 2 = split bf16 (fp32 accumulate in TMEM either way)
  int training = 0;     // 1: keep the activations backward needs and build the backward plan (bf16 or split bf16)
};

struct ParamInfo {
  std::string name;
  std::vector<long long> shape;
  long long numel = 0;
  float* d = nullptr;
  bool external = false;  // storage is a slice of a larger buffer
};

class Arena {
 public:
  size_t alloc(size_t bytes);
  void release(size_t off);
  size_t peak() const { return peak_; }
  size_t in_use() const { size_t n = 0; for (auto& b : blocks_) if (!b.free) n += b.size; return n; }
  void reset() { blocks_.clear(); end_ = 0; }
 private:
  struct Block { size_t off, size; bool free; };
  std::vector<Block> blocks_;
  size_t end_ = 0, peak_ = 0;
};

// A gradient buffer in the arena, shared by the views handed to the tensors it is the gradient of (the two halves of
// a channel concatenation); returned to the arena when the last view is dropped.
struct GradBuf { size_t off = 0; int refs = 0; bool has_cs = false; size_t cs_off = 0; };
struct GradView {
  std::shared_ptr<GradBuf> buf;
  void* ptr = nullptr;
  long long ld = 0;
  int C = 0;
  float* colsum = nullptr;  // [B][cs_ld] per-sample column sums of this view's channels (left by gn_bwd_apply), or null
  long long cs_ld = 0;
  bool valid() const { return buf != nullptr; }
};

struct Tens {
  size_t off = 0, bytes = 0;
  int C = 0, R = 0;
  long long* stats = nullptr;
  void* ptr = nullptr;
  bool live = true;   // arena block still held
  GradView grad;      // training: dL/d(this), set by the backward of its consumers
};
typedef std::shared_ptr<Tens> TensP;

class UNet {
 public:
  // dry_only: size the plan and enumerate parameters without touching the GPU (host-side tests)
  explicit UNet(const UNetConfig& cfg, bool dry_only = false);
  ~UNet();
  const std::vector<ParamInfo>& params() const { return params_; }
  // copies `numel` floats into the named parameter (src on host or device)
  void set_param(const std::string& name, const float* src, long long numel, bool src_device, cudaStream_t s);
  void get_param(const std::string& name, float* dst, long long numel, bool dst_device, cudaStream_t s);
  // after (re)loading parameters: derived vectors, constant stem field, weight packing
  void commit(cudaStream_t s);
  // x: fp32 NCDHW [B][Cin][R^3]; labels: fp32 [B]; out: fp32 NCDHW [B][Cin][R^3]
  // allow_graph: the caller promises that (x, labels, out) are the SAME buffers call after call (the sampler loop): for
  // small batches, where the ~200 launches of a step are launch-latency bound, the whole step is then captured once
  // into a CUDA graph (on a private capture stream) and replayed on `s`
  void forward(const float* x, const float* labels, float* out, int B, cudaStream_t s, bool allow_graph = false);
  // training engines only. Dropout of the next forward()/backward() pair (p = 0 disables; same seed in both).
  void set_dropout(float p, unsigned long long seed);
  // dout: fp32 NCDHW dL/d(out) of the preceding forward() (same x, labels, B). grads: flat fp32 buffer holding the
  // gradient of every parameter in table order (params()[i] at the sum of the numels before it); entries of
  // non-trainable tensors (mask, coords, pos_layer.weight) are left untouched. accumulate: += instead of =.
  // marks (optional): after `mark_steps[j]` backward launches have been enqueued (ascending), the CUDA event
  // mark_events[j] is recorded on `s` -- the hook a data-parallel host uses to start all-reducing a gradient bucket while
  // the rest of the backward pass still runs (grad_ready_step tells it after which launch a parameter's gradient is final)
  void backward(const float* dout, float* grads, int B, bool accumulate, cudaStream_t s, const int* mark_steps = nullptr,
                void* const* mark_events = nullptr, int n_marks = 0);
  int grad_ready_step(const std::string& name) const;
  long long grad_offset(const std::string& name) const;
  long long total_param_numel() const;
  int num_bwd_steps() const { return (int)bwd_steps_.size(); }
  // diagnostics: raw GroupNorm statistics of the last forward ([tensor][B][C][2] int64, 2^-24 fixed point)
  size_t stats_count() const { return stats_doubles_; }
  const long long* stats_ptr() const { return stats_base_; }
  double bwd_flops_per_sample() const { return bwd_flops_ / cfg_.max_batch; }
  std::vector<std::pair<std::string, float>> profile_backward(const float* dout, float* grads, int B, cudaStream_t s);
  double flops_per_sample() const { return flops_ / cfg_.max_batch; }
  size_t arena_bytes() const { return arena_bytes_; }
  int num_gemm_launches() const { return (int)gemms_.size(); }
  int num_steps() const { return (int)steps_.size(); }
  const UNetConfig& cfg() const { return cfg_; }
  // per-GEMM timing breakdown of one forward (ms), for profiling
  std::vector<std::pair<std::string, float>> profile(const float* x, const float* labels, float* out, int B, cudaStream_t s);

 private:
  UNetConfig cfg_;
  Precision prec_;
  bool dry_ = true;
  std::vector<ParamInfo> params_;
  std::map<std::string, int> pindex_;
  std::vector<void*> owned_;  // cudaMalloc'd buffers
  Arena arena_;
  char* arena_base_ = nullptr;
  size_t arena_bytes_ = 0;
  long long* stats_base_ = nullptr;
  size_t stats_doubles_ = 0, stats_cursor_ = 0;
  std::vector<std::unique_ptr<GemmOp>> gemms_;
  std::vector<std::unique_ptr<GemmOp>> commit_gemms_;
  struct Step { std::string name; std::function<void(cudaStream_t, int)> fn; };
  std::vector<Step> steps_, commit_steps_;
  bool committed_ = false;
  double flops_ = 0;
  // CUDA-graph replay of the forward plan (allow_graph): one instantiated graph per (x, labels, out, B)
  struct FwdGraph { const float* x; const float* labels; float* out; int B; int uses; cudaGraphExec_t exec; };
  std::vector<FwdGraph> graphs_;
  cudaStream_t capture_stream_ = nullptr;
  int graph_max_batch_ = 8;
  void drop_graphs();
  // runtime pointers
  const float* rt_x_ = nullptr;
  const float* rt_labels_ = nullptr;
  float* rt_out_ = nullptr;
  // temb
  float* temb_act_ = nullptr;
  float* dense_w_ = nullptr; float* dense_b_ = nullptr; float* dense_out_ = nullptr;
  int dense_total_ = 0, dense_cursor_ = 0;

  void build();
  float* P(const std::string& name, std::vector<long long> shape, float* external = nullptr);
  void* dmalloc(size_t bytes, bool zero = true);
  TensP new_act(int C, int R, bool stats);
  void release(TensP& t);
  Act act_of(const TensP& t) const;
  GemmOp* new_gemm(const std::string& name, bool commit_time = false);
  void add_step(const std::string& name, std::function<void(cudaStream_t, int)> fn) { if (!dry_) steps_.push_back({name, fn}); }
  struct Scratch { int S = 1; size_t off = 0; float* ptr = nullptr; bool active = false; };
  Scratch split_begin(int R, int N, int cin_total, int taps);
  void split_end(Scratch& s);
  TensP gn(const std::string& pname, const std::vector<TensP>& ins, bool silu, int drop_layer = -1);
  // ---- training plan (unet_train.cu)
  bool train_ = false;
  std::vector<std::function<void()>> tape_;  // backward emitters, pushed in forward order, run in reverse
  std::vector<Step> bwd_steps_;
  std::vector<std::unique_ptr<GemmOp>> bwd_gemms_;
  std::vector<std::unique_ptr<WgradOp>> wgrads_;
  double bwd_flops_ = 0;
  std::map<std::string, long long> goff_;
  mutable std::vector<std::string> touched_;  // parameters whose gradient offset the running backward emitter asked for
  std::map<std::string, int> grad_ready_;     // parameter -> number of backward launches after which its gradient is final
  float* rt_grads_ = nullptr; const float* rt_dout_ = nullptr; bool rt_accum_ = false;
  int rt_drop_thresh_ = 0; float rt_drop_scale_ = 1.f; unsigned long long rt_seed_ = 0;
  float* d_dense_out_ = nullptr;  // [mb][dense_total] gradient of the time-embedding projections
  int bwd_count_ = 0;  // launches of the backward plan emitted so far (counted in the dry pass too)
  void add_bwd(const std::string& name, std::function<void(cudaStream_t, int)> fn) { ++bwd_count_; if (!dry_) bwd_steps_.push_back({name, fn}); }
  void free_act(const TensP& t);
  GradView new_grad(int C, int R);
  GradView grad_view(const GradView& g, int c0, int C);
  void unref(GradView& g);
  Act act_of_grad(const GradView& g, int R) const;
  long long G(const std::string& name) const;  // offset of a parameter's gradient in the flat buffer
  struct Tmp { size_t off = 0; void* ptr = nullptr; };
  // GroupNorm backward fused into the epilogue of the data-gradient GEMM that produces dL/d(GroupNorm output):
  // filled in by the caller (which layer), completed by emit_conv_dgrad / emit_pointwise (whether it could be fused)
  struct GnFuse {
    std::string pname; std::vector<TensP> ins; bool silu = false; int drop_layer = -1;
    bool on = false; Tmp consts, part; int T = 0, bb = 1;
  };
  void gn_fuse_attach(GnFuse& f, GemmOp* g, int N, int R);
  Tmp tmp_alloc(size_t bytes);
  void tmp_free(Tmp& t);
  GemmOp* new_bwd_gemm(const std::string& name);
  void emit_colsum(const std::string& name, const GradView& t, int R, float* per, long long per_ld, long long g0, long long g1, long long g2);
  void emit_wgrad(const std::string& name, const Act& dy, const Act& x, int ksize, int stride, long long goff, const WgradOut& layout);
  GradView emit_conv_dgrad(const std::string& name, const GradView& dy, int R, const float* w, int cin_total, const GradView* addend, GnFuse* fuse = nullptr);
  GradView emit_pointwise(const std::string& name, const std::vector<Act>& srcs, const std::vector<WSrc>& ws, int N, int R, const GradView* addend, GnFuse* fuse = nullptr);
  GradView emit_gn_backward(const std::string& pname, const std::vector<TensP>& ins, const GradView& da, bool silu, int drop_layer,
                            const GradView* add0, const GradView* add1, GnFuse* fuse = nullptr);
  void tape_resblock(const std::vector<TensP>& ins, TensP a, TensP h, TensP a2, TensP out, int out_ch, int midx, int doff);
  void tape_attn(TensP x, TensP hn, TensP qkv, TensP S, TensP O, TensP out, int midx);
  void tape_downsample(TensP x, TensP out, int midx);
  void tape_upsample(TensP x, TensP up, TensP out, int midx);
  void tape_stem(TensP h0, void* Am, int Kpad, int Kpad_m);
  void tape_head(TensP h, TensP a, const std::string& gn_name, const std::string& conv_name);
  void tape_temb();
  TensP resblock(const std::vector<TensP>& ins, int out_ch, int midx);
  TensP attn(const TensP& x, int midx);
  TensP downsample(const TensP& x, int midx);
  TensP upsample(const TensP& x, int midx);
};

}  // namespace mdb

// Backward plan of the score network: what torch autograd executes for the reference's `loss.backward()`
// (lib/diffusion/losses.py:104-139) over DDPMRes64/128 (ddpm_res64.py:126-199, layers.py:573-689), emitted as a static
// list of tcgen05 data-gradient GEMMs (gemm_tc.cuh), tcgen05 weight-gradient contractions (wgrad_tc.cuh) and
// bandwidth kernels (backward.cu). Every forward builder records an emitter on a tape; build() runs the tape in
// reverse, so tensor lifetimes of the whole forward+backward step are packed into one arena by the same first-fit
// planner as the inference engine.
//
// Operand modes: bf16, or split bf16 (kBF16X3: every activation, gradient and scratch operand is a (hi, lo) pair of
// bf16 tensors in the row layout of gemm_host.h, forward and backward alike, for fp32-class gradients). Pitches handed
// between emitters stay logical; byte sizes are multiplied by parts(prec_).
#include "unet.h"
#include <cmath>
#include <cstdlib>

namespace mdb {

// ------------------------------------------------------------------ plumbing
void UNet::free_act(const TensP& t) {
  if (t && t->live) { arena_.release(t->off); t->live = false; }
}

GradView UNet::new_grad(int C, int R) {
  GradView g;
  g.buf = std::make_shared<GradBuf>();
  g.buf->off = arena_.alloc((size_t)cfg_.max_batch * R * R * R * C * esize(prec_) * parts(prec_));
  g.buf->refs = 1;
  g.ptr = dry_ ? nullptr : arena_base_ + g.buf->off;
  g.ld = C; g.C = C;
  return g;
}

GradView UNet::grad_view(const GradView& g, int c0, int C) {
  GradView v = g;
  v.buf->refs++;
  // (X3: the lo parts of the view sit one logical row (ld) behind its hi parts, so this offsets both halves)
  v.ptr = dry_ ? nullptr : (char*)g.ptr + (size_t)c0 * esize(prec_);
  v.C = C;
  if (g.colsum) v.colsum = g.colsum + c0;
  return v;
}

void UNet::unref(GradView& g) {
  if (!g.buf) return;
  if (--g.buf->refs == 0) {
    arena_.release(g.buf->off);
    if (g.buf->has_cs) arena_.release(g.buf->cs_off);
  }
  g.buf.reset();
  g.ptr = nullptr;
  g.colsum = nullptr;
}

Act UNet::act_of_grad(const GradView& g, int R) const {
  Act a;
  a.ptr = g.ptr; a.C = g.C; a.ld = g.ld; a.X = a.Y = a.Z = R; a.B = cfg_.max_batch;
  return a;
}

long long UNet::G(const std::string& name) const {
  touched_.push_back(name);
  if (dry_) return 0;
  auto it = goff_.find(name);
  if (it == goff_.end()) throw std::runtime_error("mdb: no gradient slot for " + name);
  return it->second;
}
int UNet::grad_ready_step(const std::string& name) const {
  if (goff_.find(name) == goff_.end()) throw std::runtime_error("mdb: unknown parameter " + name);
  auto it = grad_ready_.find(name);
  return it == grad_ready_.end() ? 0 : it->second;  // never written (mask, coords, pos_layer.weight): final from the start
}
long long UNet::grad_offset(const std::string& name) const {
  auto it = goff_.find(name);
  if (it == goff_.end()) throw std::runtime_error("mdb: unknown parameter " + name);
  return it->second;
}
long long UNet::total_param_numel() const {
  long long n = 0;
  for (auto& p : params_) n += p.numel;
  return n;
}

UNet::Tmp UNet::tmp_alloc(size_t bytes) {
  Tmp t;
  t.off = arena_.alloc(bytes ? bytes : 16);
  t.ptr = dry_ ? nullptr : arena_base_ + t.off;
  return t;
}
void UNet::tmp_free(Tmp& t) { arena_.release(t.off); t.ptr = nullptr; }

GemmOp* UNet::new_bwd_gemm(const std::string& name) {
  auto g = std::make_unique<GemmOp>();
  g->name = name;
  GemmOp* raw = g.get();
  bwd_gemms_.push_back(std::move(g));
  return raw;
}

void UNet::set_dropout(float p, unsigned long long seed) {
  if (p < 0.f || p >= 1.f) throw std::runtime_error("mdb: dropout probability out of range");
  rt_drop_thresh_ = (int)std::lround((double)p * 65536.0);
  rt_drop_scale_ = p > 0.f ? 1.f / (1.f - p) : 1.f;
  rt_seed_ = seed;
}

void UNet::backward(const float* dout, float* grads, int B, bool accumulate, cudaStream_t s, const int* mark_steps,
                    void* const* mark_events, int n_marks) {
  if (!train_) throw std::runtime_error("mdb: backward() needs an engine created with training = 1");
  if (!committed_) throw std::runtime_error("mdb: parameters changed, call commit() before backward()");
  if (B < 1 || B > cfg_.max_batch) throw std::runtime_error("mdb: batch out of range");
  for (int j = 1; j < n_marks; ++j)
    if (mark_steps[j] < mark_steps[j - 1]) throw std::runtime_error("mdb: backward marks must be in ascending step order");
  rt_dout_ = dout; rt_grads_ = grads; rt_accum_ = accumulate;
  int mi = 0;
  auto fire = [&](int done) {
    while (mi < n_marks && mark_steps[mi] <= done) MDB_CUDA_CHECK(cudaEventRecord((cudaEvent_t)mark_events[mi++], s));
  };
  fire(0);
  for (size_t i = 0; i < bwd_steps_.size(); ++i) {
    bwd_steps_[i].fn(s, B);
    fire((int)i + 1);
  }
  fire(1 << 30);
}

std::vector<std::pair<std::string, float>> UNet::profile_backward(const float* dout, float* grads, int B, cudaStream_t s) {
  if (!train_) throw std::runtime_error("mdb: profile_backward() needs a training engine");
  rt_dout_ = dout; rt_grads_ = grads; rt_accum_ = false;
  std::vector<std::pair<std::string, float>> res;
  std::vector<cudaEvent_t> ev(bwd_steps_.size() + 1);
  for (auto& e : ev) MDB_CUDA_CHECK(cudaEventCreate(&e));
  MDB_CUDA_CHECK(cudaEventRecord(ev[0], s));
  for (size_t i = 0; i < bwd_steps_.size(); ++i) {
    bwd_steps_[i].fn(s, B);
    MDB_CUDA_CHECK(cudaEventRecord(ev[i + 1], s));
  }
  MDB_CUDA_CHECK(cudaStreamSynchronize(s));
  for (size_t i = 0; i < bwd_steps_.size(); ++i) {
    float ms = 0;
    MDB_CUDA_CHECK(cudaEventElapsedTime(&ms, ev[i], ev[i + 1]));
    res.push_back({bwd_steps_[i].name, ms});
  }
  for (auto& e : ev) cudaEventDestroy(e);
  return res;
}

// ------------------------------------------------------------------ emit helpers
// per[b][c] = sum_v t[b][v][c] (optional) and up to three parameter gradients (offsets, -1 = none) += sum_b per[b][c]
void UNet::emit_colsum(const std::string& name, const GradView& t, int R, float* per, long long per_ld, long long g0,
                       long long g1, long long g2) {
  // when the producing GroupNorm-backward kernel already left per-sample column sums, only the batch sum remains
  const bool have = t.buf && t.buf->has_cs;
  Tmp part = tmp_alloc(have ? 16 : (size_t)kBwdPartRows(cfg_.max_batch) * t.C * sizeof(float));
  if (!dry_) {
    ColsumArgs a{};
    a.t = t.ptr; a.ld = t.ld; a.C = t.C; a.voxels = (long long)R * R * R;
    a.part = (float*)part.ptr; a.per = per; a.per_ld = per_ld;
    a.from_per = t.colsum; a.from_ld = t.cs_ld;
    a.x3 = prec_ == kBF16X3 ? 1 : 0;
    add_bwd(name, [=](cudaStream_t s, int B) {
      ColsumArgs c = a;
      c.total0 = g0 >= 0 ? rt_grads_ + g0 : nullptr;
      c.total1 = g1 >= 0 ? rt_grads_ + g1 : nullptr;
      c.total2 = g2 >= 0 ? rt_grads_ + g2 : nullptr;
      c.accumulate = rt_accum_ ? 1 : 0;
      launch_colsum(c, B, s);
    });
  }
  tmp_free(part);
}

// G[tap][m][n] = sum_p dy[p][m] x[p+tap][n] scattered to the parameter gradient at `goff` with `layout` strides
void UNet::emit_wgrad(const std::string& name, const Act& dy, const Act& x, int ksize, int stride, long long goff,
                      const WgradOut& layout) {
  const WgradPlan pl = plan_wgrad(dy.X, dy.Y, dy.Z, dy.B, dy.C, x.C, ksize, stride);
  Tmp sc = tmp_alloc(pl.scratch_bytes);
  if (!dry_) {
    auto op = std::make_unique<WgradOp>();
    op->name = name;
    op->init(dy, x, ksize, stride, layout, (float*)sc.ptr, prec_ == kBF16X3);
    WgradOp* raw = op.get();
    wgrads_.push_back(std::move(op));
    const bool fixed = dy.B == 1 && cfg_.max_batch != 1;  // batch-reduced operand (mask_layer)
    add_bwd(name, [=](cudaStream_t s, int B) { raw->launch(s, fixed ? 1 : B, rt_accum_, rt_grads_ + goff); });
  }
  tmp_free(sc);
}

// data gradient of a stride-1 3^3 convolution: [C = cin_total] = conv(dy, W^T mirrored) (+ addend)
// MDB_GNB=0 keeps the two-pass GroupNorm backward everywhere (A/B comparisons; tests compare both paths under dropout)
static bool gnb_enabled() {
  const char* e = getenv("MDB_GNB");
  return !(e && e[0] == '0');
}

// Sizes and attaches the GroupNorm-backward epilogue of a data-gradient GEMM (same decisions in the sizing pass, where
// g == nullptr, and the real pass).
void UNet::gn_fuse_attach(GnFuse& f, GemmOp* g, int N, int R) {
  const int mb = cfg_.max_batch;
  const Geometry geo = pick_geometry(R, R, R);
  f.T = ((R + geo.bx - 1) / geo.bx) * ((R + geo.by - 1) / geo.by) * ((R + geo.bz - 1) / geo.bz);
  f.bb = geo.bb;
  const long long rows = 1LL * f.T * ((mb + geo.bb - 1) / geo.bb) * geo.bb;
  f.consts = tmp_alloc((size_t)mb * N * 4 * sizeof(float));
  f.part = tmp_alloc((size_t)rows * N * 2 * sizeof(float));
  f.on = true;
  if (dry_) return;
  GnBwdArgs a{};
  a.C0 = f.ins[0]->C; a.C1 = f.ins.size() > 1 ? f.ins[1]->C : 0;
  a.stats0 = f.ins[0]->stats; a.stats1 = f.ins.size() > 1 ? f.ins[1]->stats : nullptr;
  a.gamma = P(f.pname + ".weight", {N}); a.beta = P(f.pname + ".bias", {N});
  a.voxels = (long long)R * R * R; a.groups = 32; a.eps = 1e-6f;
  float* cp = (float*)f.consts.ptr;
  add_bwd("gn_consts:" + f.pname, [a, cp](cudaStream_t s, int B) { launch_gn_consts(a, cp, B, s); });
  g->set_gn_backward(f.ins[0]->ptr, f.ins[0]->C, f.ins[0]->C, f.ins.size() > 1 ? f.ins[1]->ptr : nullptr,
                     f.ins.size() > 1 ? f.ins[1]->C : 0, f.consts.ptr, f.silu ? 1 : 0, (float*)f.part.ptr);
  if (g->gnb_tiles_per_batch_tile() != f.T || g->gnb_bb() != f.bb) throw std::runtime_error("mdb: GroupNorm-backward tile plan mismatch");
}

GradView UNet::emit_conv_dgrad(const std::string& name, const GradView& dy, int R, const float* w, int cin_total,
                               const GradView* addend, GnFuse* fuse) {
  GradView dx = new_grad(cin_total, R);
  const bool can_split = !addend || addend->ld == cin_total;
  Scratch sp;
  if (can_split) sp = split_begin(R, cin_total, dy.C, 27);
  const bool fused = fuse && gnb_enabled() && !addend && sp.S <= 1 && cin_total % 32 == 0;
  GemmOp* g = nullptr;
  if (!dry_) {
    g = new_bwd_gemm(name);
    g->set_output(prec_, R, R, R, cfg_.max_batch, cin_total, dx.ptr, cin_total, false);
    g->add_conv_dgrad(act_of_grad(dy, R), w, cin_total, 3);
    if (addend) g->set_residual(addend->ptr, addend->ld, (long long)R * R * R * addend->ld, false);
    g->enable_splits(sp.S, sp.ptr);
  }
  if (fused) gn_fuse_attach(*fuse, g, cin_total, R);
  if (!dry_) {
    g->finalize(0, false);
    const int dl = fused ? fuse->drop_layer : -1;
    add_bwd(name, [g, this, dl](cudaStream_t s, int B) {
      if (dl >= 0) {
        g->rt_drop_thresh = rt_drop_thresh_; g->rt_drop_scale = rt_drop_scale_;
        g->rt_seed = rt_seed_ + 0x632BE59BD9B4E019ull * (unsigned long long)(dl + 1);
      }
      g->launch(s, B);
    });
  }
  split_end(sp);
  return dx;
}

// [N] = sum_i srcs[i] . ws[i]  (1x1x1 products accumulated in one TMEM accumulator) (+ addend)
GradView UNet::emit_pointwise(const std::string& name, const std::vector<Act>& srcs, const std::vector<WSrc>& ws, int N, int R,
                              const GradView* addend, GnFuse* fuse) {
  GradView dx = new_grad(N, R);
  const bool fused = fuse && gnb_enabled() && !addend && N % 32 == 0;
  GemmOp* g = nullptr;
  if (!dry_) {
    g = new_bwd_gemm(name);
    g->set_output(prec_, R, R, R, cfg_.max_batch, N, dx.ptr, N, false);
    for (size_t i = 0; i < srcs.size(); ++i) g->add_pointwise_w({srcs[i]}, &ws[i]);
    if (addend) g->set_residual(addend->ptr, addend->ld, (long long)R * R * R * addend->ld, false);
  }
  if (fused) gn_fuse_attach(*fuse, g, N, R);
  if (!dry_) {
    g->finalize(0, false);
    add_bwd(name, [g](cudaStream_t s, int B) { g->launch(s, B); });
  }
  return dx;
}

GradView UNet::emit_gn_backward(const std::string& pname, const std::vector<TensP>& ins, const GradView& da, bool silu,
                                int drop_layer, const GradView* add0, const GradView* add1, GnFuse* fuse) {
  int C = 0;
  for (auto& t : ins) C += t->C;
  const int R = ins[0]->R, mb = cfg_.max_batch;
  float* gamma = P(pname + ".weight", {C});
  float* beta = P(pname + ".bias", {C});
  if (da.ld != C) throw std::runtime_error("mdb: GroupNorm backward needs a dense upstream gradient");
  const bool fused = fuse && fuse->on;  // `da` already holds dy and the GEMM left per-tile partials: no pass 1
  Tmp part = tmp_alloc(fused ? 16 : (size_t)kBwdPartRows(mb) * C * 2 * sizeof(float));
  Tmp sums = tmp_alloc((size_t)mb * C * 2 * sizeof(float));
  GradView dx = new_grad(C, R);
  // by-product of the apply pass: per-(sample, channel) sums of dx, kept with the buffer for the bias gradients of
  // whichever op produced the tensor this is the gradient of
  dx.buf->has_cs = true;
  dx.buf->cs_off = arena_.alloc((size_t)mb * C * sizeof(float));
  dx.colsum = dry_ ? nullptr : reinterpret_cast<float*>(arena_base_ + dx.buf->cs_off);
  dx.cs_ld = C;
  Tmp cs_part = tmp_alloc((size_t)kBwdPartRows(mb) * C * sizeof(float));
  if (!dry_) {
    GnBwdArgs a{};
    a.x0 = ins[0]->ptr; a.C0 = ins[0]->C; a.ld0 = ins[0]->C;
    a.x1 = ins.size() > 1 ? ins[1]->ptr : nullptr; a.C1 = ins.size() > 1 ? ins[1]->C : 0; a.ld1 = a.C1;
    a.stats0 = ins[0]->stats; a.stats1 = ins.size() > 1 ? ins[1]->stats : nullptr;
    a.gamma = gamma; a.beta = beta; a.da = da.ptr;
    a.voxels = (long long)R * R * R; a.silu = silu ? 1 : 0; a.groups = 32; a.eps = 1e-6f;
    a.part = (float*)part.ptr; a.sums = (float*)sums.ptr;
    a.dx = dx.ptr;
    a.add0 = add0 ? add0->ptr : nullptr; a.add0_ld = add0 ? add0->ld : 0;
    a.add1 = add1 ? add1->ptr : nullptr; a.add1_ld = add1 ? add1->ld : 0;
    a.cs_part = (float*)cs_part.ptr; a.cs_per = dx.colsum;
    a.x3 = prec_ == kBF16X3 ? 1 : 0;
    const long long gw = G(pname + ".weight"), gb = G(pname + ".bias");
    auto with_rt = [this, a, gw, gb, drop_layer]() {
      GnBwdArgs c = a;
      if (drop_layer >= 0) {
        c.drop_thresh = rt_drop_thresh_; c.drop_scale = rt_drop_scale_;
        c.seed = rt_seed_ + 0x632BE59BD9B4E019ull * (unsigned long long)(drop_layer + 1);
      }
      c.dgamma = rt_grads_ + gw; c.dbeta = rt_grads_ + gb; c.accumulate = rt_accum_ ? 1 : 0;
      return c;
    };
    if (fused) {
      const float* tp = (const float*)fuse->part.ptr; const int T = fuse->T, bb = fuse->bb;
      add_bwd("gnb_tile_reduce:" + pname, [with_rt, tp, T, bb](cudaStream_t s, int B) { launch_gnb_tile_reduce(with_rt(), tp, T, bb, B, s); });
    } else {
      add_bwd("gn_bwd_reduce:" + pname, [with_rt](cudaStream_t s, int B) { launch_gn_bwd_reduce(with_rt(), B, s); });
    }
    add_bwd("gn_bwd_apply:" + pname, [with_rt](cudaStream_t s, int B) { launch_gn_bwd_apply(with_rt(), B, s); });
  }
  tmp_free(part);
  tmp_free(sums);
  tmp_free(cs_part);
  if (fused) { tmp_free(fuse->consts); tmp_free(fuse->part); fuse->on = false; }
  return dx;
}

static WgradOut oidhw_layout(int cin_total) {
  WgradOut o;
  o.sm = 27LL * cin_total; o.sn = 27; o.st = 1;
  return o;
}
static WgradOut in_out_layout(int n_out) {  // NIN W[in][out]: G[m = out][n = in]
  WgradOut o;
  o.sm = 1; o.sn = n_out; o.st = 0;
  return o;
}

// ------------------------------------------------------------------ ResnetBlockDDPM (layers.py:646-689)
void UNet::tape_resblock(const std::vector<TensP>& ins, TensP a, TensP h, TensP a2, TensP out, int out_ch, int midx, int doff) {
  tape_.push_back([=]() {
    const std::string pre = "all_modules." + std::to_string(midx) + ".";
    const std::string nm = "res" + std::to_string(midx);
    int Cin = 0;
    for (auto& t : ins) Cin += t->C;
    const int R = out->R, tdim = 4 * cfg_.nf;
    const bool nin = Cin != out_ch;
    float* w0 = P(pre + "Conv_0.weight", {});
    float* w1 = P(pre + "Conv_1.weight", {});
    float* wn = nin ? P(pre + "NIN_0.W", {}) : nullptr;
    free_act(out);
    GradView dO = out->grad;
    if (!dO.valid()) throw std::runtime_error("mdb: " + nm + " has no upstream gradient");
    // Conv_1 bias (the folded NIN_0 bias sees the same sum)
    emit_colsum(nm + ".conv1.dbias", dO, R, nullptr, 0, G(pre + "Conv_1.bias"), nin ? G(pre + "NIN_0.b") : -1, -1);
    emit_wgrad(nm + ".conv1.wgrad", act_of_grad(dO, R), act_of(a2), 3, 1, G(pre + "Conv_1.weight"), oidhw_layout(out_ch));
    if (nin) {
      int coff = 0;
      for (auto& t : ins) {
        emit_wgrad(nm + ".nin.wgrad", act_of_grad(dO, R), act_of(t), 1, 1, G(pre + "NIN_0.W") + (long long)coff * out_ch, in_out_layout(out_ch));
        coff += t->C;
      }
    }
    GnFuse f1; f1.pname = pre + "GroupNorm_1"; f1.ins = {h}; f1.silu = true; f1.drop_layer = midx;
    GradView da2 = emit_conv_dgrad(nm + ".conv1.dgrad", dO, R, w1, out_ch, nullptr, &f1);
    free_act(a2);
    GradView dh = emit_gn_backward(pre + "GroupNorm_1", {h}, da2, true, midx, nullptr, nullptr, &f1);
    unref(da2);
    // Conv_0 bias and the time-embedding projection: h += Dense_0(act(temb))[:, :, None, None, None]
    emit_colsum(nm + ".conv0.dbias", dh, R, dry_ ? nullptr : d_dense_out_ + doff, dense_total_, G(pre + "Conv_0.bias"), -1, -1);
    if (!dry_) {
      const float* dd = d_dense_out_ + doff; const long long dt = dense_total_; const float* ta = temb_act_;
      const long long gw = G(pre + "Dense_0.weight"), gb = G(pre + "Dense_0.bias");
      add_bwd(nm + ".dense.wgrad", [=](cudaStream_t s, int B) {
        launch_outer_sum(dd, dt, ta, tdim, rt_grads_ + gw, rt_grads_ + gb, B, out_ch, tdim, rt_accum_ ? 1 : 0, s);
      });
    }
    emit_wgrad(nm + ".conv0.wgrad", act_of_grad(dh, R), act_of(a), 3, 1, G(pre + "Conv_0.weight"), oidhw_layout(Cin));
    free_act(a);
    GnFuse f0; f0.pname = pre + "GroupNorm_0"; f0.ins = ins; f0.silu = true; f0.drop_layer = -1;
    GradView da = emit_conv_dgrad(nm + ".conv0.dgrad", dh, R, w0, Cin, nullptr, &f0);
    unref(dh);
    free_act(h);
    // shortcut: identity -> dO itself; NIN -> dO . W^T
    GradView sc;
    if (nin) sc = emit_pointwise(nm + ".nin.dgrad", {act_of_grad(dO, R)}, {WSrc{wn, (long long)out_ch, 1, 0, out_ch}}, Cin, R, nullptr);
    GradView prev = ins.size() == 1 ? ins[0]->grad : GradView{};
    GradView dx = emit_gn_backward(pre + "GroupNorm_0", ins, da, true, -1, nin ? &sc : &dO, prev.valid() ? &prev : nullptr, &f0);
    unref(da);
    if (nin) unref(sc);
    unref(out->grad);
    if (prev.valid()) unref(ins[0]->grad);
    if (ins.size() == 1) {
      ins[0]->grad = dx;
    } else {
      ins[0]->grad = grad_view(dx, 0, ins[0]->C);
      ins[1]->grad = grad_view(dx, ins[0]->C, ins[1]->C);
      unref(dx);
    }
  });
}

// ------------------------------------------------------------------ AttnBlock (layers.py:585-608)
void UNet::tape_attn(TensP x, TensP hn, TensP qkv, TensP S, TensP O, TensP out, int midx) {
  tape_.push_back([=]() {
    const std::string pre = "all_modules." + std::to_string(midx) + ".";
    const std::string nm = "attn" + std::to_string(midx);
    const int C = x->C, R = x->R, mb = cfg_.max_batch;
    const int V = R * R * R;
    float* W[4];
    for (int i = 0; i < 4; ++i) W[i] = P(pre + "NIN_" + std::to_string(i) + ".W", {});
    free_act(out);
    GradView dO = out->grad;
    if (!dO.valid()) throw std::runtime_error("mdb: " + nm + " has no upstream gradient");
    // out = x + NIN_3(O)
    emit_colsum(nm + ".nin3.dbias", dO, R, nullptr, 0, G(pre + "NIN_3.b"), -1, -1);
    emit_wgrad(nm + ".nin3.wgrad", act_of_grad(dO, R), act_of(O), 1, 1, G(pre + "NIN_3.W"), in_out_layout(C));
    free_act(O);
    GradView dOo = emit_pointwise(nm + ".nin3.dgrad", {act_of_grad(dO, R)}, {WSrc{W[3], (long long)C, 1, 0, C}}, C, R, nullptr);
    auto mat = [&](void* ptr, int K, long long ld) {  // a [V][K] operand matrix per sample
      Act a; a.ptr = ptr; a.C = K; a.ld = ld; a.X = V; a.Y = 1; a.Z = 1; a.B = mb;
      return a;
    };
    const float alpha = 1.0f / std::sqrt((float)C);
    const bool x3 = prec_ == kBF16X3;
    const size_t pp = parts(prec_);
    // transposed copy out[b][c][v] = in[b][v][c0 + c] of an operand matrix; X3: rows [ld hi | ld lo] -> [V hi | V lo]
    auto transpose = [x3, V](const void* in, long long ld, int c0, void* out, int B, int C_, cudaStream_t s) {
      launch_transpose_vc_rows(in, ld, c0, out, B, V, C_, x3 ? 1 : 0, s);
    };
    // P and dS: probabilities / logit gradients in the activation dtype at the start of rows of V fp32 slots -- a logical
    // pitch of 2V bf16, or V for X3 (whose [V hi | V lo] rows fill the slots)
    const long long sld = x3 ? V : 2LL * V;
    GradView dqkv = new_grad(3 * C, R);
    // dP[q][k] = dOo[q][:] . v[k][:]   (fp32, softmax backward then runs in place)
    Tmp dS = tmp_alloc((size_t)mb * V * V * 4);
    if (!dry_) {
      GemmOp* g = new_bwd_gemm(nm + ".dP");
      g->set_output_strided(prec_, V, 1, 1, mb, V, dS.ptr, V, 0, 0, (long long)V * V, true);
      g->add_pointwise({mat(dOo.ptr, C, C)}, nullptr, true);
      g->set_b_activation((char*)qkv->ptr + (size_t)2 * C * 2, C, V, mb, 3 * C, (long long)V * 3 * C);
      g->finalize(0, false);
      add_bwd(g->name, [g](cudaStream_t s, int B) { g->launch(s, B); });
    }
    // dv[k][c] = sum_q P[q][k] dOo[q][c]
    Tmp PT = tmp_alloc((size_t)mb * V * V * 2 * pp);
    Tmp dOT = tmp_alloc((size_t)mb * C * V * 2 * pp);
    if (!dry_) {
      const void* sp = S->ptr; void* pt = PT.ptr; const void* dop = dOo.ptr; void* dot = dOT.ptr;
      add_bwd(nm + ".PT", [=](cudaStream_t s, int B) {
        transpose(sp, sld, 0, pt, B, V, s);
        transpose(dop, C, 0, dot, B, C, s);
      });
      GemmOp* g = new_bwd_gemm(nm + ".dv");
      g->set_output_strided(prec_, V, 1, 1, mb, C, (char*)dqkv.ptr + (size_t)2 * C * 2, 3 * C, 0, 0, (long long)V * 3 * C, false);
      g->add_pointwise({mat(PT.ptr, V, V)}, nullptr, true);
      g->set_b_activation(dOT.ptr, V, C, mb, V, (long long)C * V);
      g->finalize(0, false);
      add_bwd(g->name, [g](cudaStream_t s, int B) { g->launch(s, B); });
      float* dsp = (float*)dS.ptr; const float* Pp = (const float*)S->ptr;
      const int xm = x3 ? 1 : 0;
      add_bwd(nm + ".softmax_bwd", [=](cudaStream_t s, int B) { launch_softmax_bwd_rows(Pp, dsp, (long long)B * V, V, xm, s); });
    }
    tmp_free(PT);
    tmp_free(dOT);
    unref(dOo);
    free_act(S);
    // dq = alpha dS . k ; dk = alpha dS^T . q
    Tmp kT = tmp_alloc((size_t)mb * C * V * 2 * pp);
    Tmp qT = tmp_alloc((size_t)mb * C * V * 2 * pp);
    Tmp dST = tmp_alloc((size_t)mb * V * V * 2 * pp);
    if (!dry_) {
      const void* qp = qkv->ptr; void* ktp = kT.ptr; void* qtp = qT.ptr; const void* dsp = dS.ptr; void* dstp = dST.ptr;
      add_bwd(nm + ".kT", [=](cudaStream_t s, int B) {
        transpose(qp, 3 * C, C, ktp, B, C, s);
        transpose(qp, 3 * C, 0, qtp, B, C, s);
        transpose(dsp, sld, 0, dstp, B, V, s);
      });
      GemmOp* g = new_bwd_gemm(nm + ".dq");
      g->set_output_strided(prec_, V, 1, 1, mb, C, dqkv.ptr, 3 * C, 0, 0, (long long)V * 3 * C, false);
      g->add_pointwise({mat(dS.ptr, V, sld)}, nullptr, true);
      g->set_b_activation(kT.ptr, V, C, mb, V, (long long)C * V);
      g->set_alpha(alpha);
      g->finalize(0, false);
      add_bwd(g->name, [g](cudaStream_t s, int B) { g->launch(s, B); });
      GemmOp* g2 = new_bwd_gemm(nm + ".dk");
      g2->set_output_strided(prec_, V, 1, 1, mb, C, (char*)dqkv.ptr + (size_t)C * 2, 3 * C, 0, 0, (long long)V * 3 * C, false);
      g2->add_pointwise({mat(dST.ptr, V, V)}, nullptr, true);
      g2->set_b_activation(qT.ptr, V, C, mb, V, (long long)C * V);
      g2->set_alpha(alpha);
      g2->finalize(0, false);
      add_bwd(g2->name, [g2](cudaStream_t s, int B) { g2->launch(s, B); });
    }
    tmp_free(kT);
    tmp_free(qT);
    tmp_free(dST);
    tmp_free(dS);
    // q, k, v = NIN_{0,1,2}(hn)
    std::vector<Act> parts;
    std::vector<WSrc> wsv;
    for (int i = 0; i < 3; ++i) {
      GradView part = grad_view(dqkv, i * C, C);
      emit_colsum(nm + ".nin" + std::to_string(i) + ".dbias", part, R, nullptr, 0, G(pre + "NIN_" + std::to_string(i) + ".b"), -1, -1);
      emit_wgrad(nm + ".nin" + std::to_string(i) + ".wgrad", act_of_grad(part, R), act_of(hn), 1, 1, G(pre + "NIN_" + std::to_string(i) + ".W"), in_out_layout(C));
      parts.push_back(act_of_grad(part, R));
      wsv.push_back(WSrc{W[i], (long long)C, 1, 0, C});
      unref(part);
    }
    free_act(hn);
    free_act(qkv);
    GnFuse fa; fa.pname = pre + "GroupNorm_0"; fa.ins = {x}; fa.silu = false; fa.drop_layer = -1;
    GradView dhn = emit_pointwise(nm + ".qkv.dgrad", parts, wsv, C, R, nullptr, &fa);
    unref(dqkv);
    GradView prev = x->grad;
    GradView dx = emit_gn_backward(pre + "GroupNorm_0", {x}, dhn, false, -1, &dO, prev.valid() ? &prev : nullptr, &fa);
    unref(dhn);
    unref(out->grad);
    if (prev.valid()) unref(x->grad);
    x->grad = dx;
  });
}

// ------------------------------------------------------------------ Downsample (layers.py:626-643)
void UNet::tape_downsample(TensP x, TensP out, int midx) {
  tape_.push_back([=]() {
    const std::string pre = "all_modules." + std::to_string(midx) + ".";
    const std::string nm = "down" + std::to_string(midx);
    const int C = x->C, Ro = out->R, Ri = x->R;
    float* w = P(pre + "Conv_0.weight", {});
    free_act(out);
    GradView dO = out->grad;
    if (!dO.valid() || dO.ld != C) throw std::runtime_error("mdb: " + nm + " needs a dense upstream gradient");
    emit_colsum(nm + ".dbias", dO, Ro, nullptr, 0, G(pre + "Conv_0.bias"), -1, -1);
    emit_wgrad(nm + ".wgrad", act_of_grad(dO, Ro), act_of(x), 3, 2, G(pre + "Conv_0.weight"), oidhw_layout(C));
    // transposed stride-2 convolution = zero-stuffed dY (odd sites) convolved with the mirrored, transposed kernel
    GradView z = new_grad(C, Ri);
    if (!dry_) {
      const void* src = dO.ptr; void* dst = z.ptr;
      const int Cp = C * parts(prec_);  // X3: whole (hi, lo) rows
      add_bwd(nm + ".zero_stuff", [=](cudaStream_t s, int B) { launch_zero_stuff2x(src, dst, B, Ro, Cp, s); });
    }
    GradView prev = x->grad;
    GradView dx = emit_conv_dgrad(nm + ".dgrad", z, Ri, w, C, prev.valid() ? &prev : nullptr);
    unref(z);
    unref(out->grad);
    if (prev.valid()) unref(x->grad);
    x->grad = dx;
  });
}

// ------------------------------------------------------------------ Upsample (layers.py:611-623)
void UNet::tape_upsample(TensP x, TensP up, TensP out, int midx) {
  tape_.push_back([=]() {
    const std::string pre = "all_modules." + std::to_string(midx) + ".";
    const std::string nm = "up" + std::to_string(midx);
    const int C = x->C, R = out->R;
    float* w = P(pre + "Conv_0.weight", {});
    free_act(out);
    GradView dO = out->grad;
    if (!dO.valid()) throw std::runtime_error("mdb: " + nm + " has no upstream gradient");
    emit_colsum(nm + ".dbias", dO, R, nullptr, 0, G(pre + "Conv_0.bias"), -1, -1);
    emit_wgrad(nm + ".wgrad", act_of_grad(dO, R), act_of(up), 3, 1, G(pre + "Conv_0.weight"), oidhw_layout(C));
    free_act(up);
    GradView dup = emit_conv_dgrad(nm + ".dgrad", dO, R, w, C, nullptr);
    unref(out->grad);
    GradView dx = new_grad(C, x->R);
    if (!dry_) {
      const void* src = dup.ptr; void* dst = dx.ptr; const int r = x->R; const int xm = prec_ == kBF16X3 ? 1 : 0;
      add_bwd(nm + ".downsum", [=](cudaStream_t s, int B) { launch_downsum2x(src, dst, B, r, C, xm, s); });
    }
    unref(dup);
    if (x->grad.valid()) throw std::runtime_error("mdb: upsample input already has a gradient");
    x->grad = dx;
  });
}

// ------------------------------------------------------------------ stem (ddpm_res64.py:148 / ddpm_res128.py:159-162)
void UNet::tape_stem(TensP h0, void* Am, int Kpad, int Kpad_m) {
  tape_.push_back([=]() {
    const int nf = cfg_.nf, R0 = cfg_.image_size, Cin = cfg_.num_channels, k = cfg_.stem_ksize, T = k * k * k;
    const long long V0 = (long long)R0 * R0 * R0;
    free_act(h0);
    GradView dh = h0->grad;
    if (!dh.valid() || dh.ld != nf) throw std::runtime_error("mdb: stem needs a dense upstream gradient");
    // h0 = conv(x) + b + pos_layer.bias + mask_layer(mask): the three biases receive the same column sum
    emit_colsum("stem.dbias", dh, R0, nullptr, 0, G("all_modules.2.bias"), cfg_.use_pos_bias ? G("pos_layer.bias") : -1, G("mask_layer.bias"));
    // stem weight: dW[co][ci*T + tap] = sum_v dh[v][co] im2col(x)[v][ci*T + tap]  (im2col recomputed)
    const int mode = (int)prec_;
    Tmp A0 = tmp_alloc((size_t)cfg_.max_batch * V0 * Kpad * 2 * parts(prec_));
    if (!dry_) {
      void* a0 = A0.ptr;
      add_bwd("stem.im2col", [=](cudaStream_t s, int B) { launch_im2col(rt_x_, a0, B, Cin, R0, k, Kpad, mode, s); });
    }
    {
      Act xa; xa.ptr = A0.ptr; xa.C = Kpad; xa.X = xa.Y = xa.Z = R0; xa.B = cfg_.max_batch;
      WgradOut o; o.sm = (long long)Cin * T; o.sn = 1; o.st = 0; o.n_valid = Cin * T;
      emit_wgrad("stem.wgrad", act_of_grad(dh, R0), xa, 1, 1, G("all_modules.2.weight"), o);
    }
    tmp_free(A0);
    // mask_layer weight: the mask is shared by the batch -> reduce dh over the batch first
    Tmp hs = tmp_alloc((size_t)V0 * nf * 2 * parts(prec_));
    if (!dry_) {
      const void* src = dh.ptr; void* dst = hs.ptr; const int xm = prec_ == kBF16X3 ? 1 : 0;
      add_bwd("stem.batch_sum", [=](cudaStream_t s, int B) { launch_batch_sum(src, dst, B, V0 * nf, nf, xm, s); });
    }
    {
      Act da; da.ptr = hs.ptr; da.C = nf; da.X = da.Y = da.Z = R0; da.B = 1;
      Act xa; xa.ptr = Am; xa.C = Kpad_m; xa.X = xa.Y = xa.Z = R0; xa.B = 1;
      WgradOut o; o.sm = T; o.sn = 1; o.st = 0; o.n_valid = T;
      emit_wgrad("mask_layer.wgrad", da, xa, 1, 1, G("mask_layer.weight"), o);
    }
    tmp_free(hs);
    unref(h0->grad);
  });
}

// ------------------------------------------------------------------ head: GroupNorm -> SiLU -> conv(nf -> channels)
void UNet::tape_head(TensP h, TensP a, const std::string& gn_name, const std::string& conv_name) {
  tape_.push_back([=]() {
    const int nf = cfg_.nf, R0 = cfg_.image_size, Cin = cfg_.num_channels, k = cfg_.stem_ksize, T = k * k * k;
    const long long V0 = (long long)R0 * R0 * R0;
    float* hw = P(conv_name + ".weight", {});
    if (!dry_) {
      const long long gb = G(conv_name + ".bias");
      add_bwd("head.dbias", [=](cudaStream_t s, int B) { launch_rowsum_nc(rt_dout_, rt_grads_ + gb, B, Cin, V0, rt_accum_ ? 1 : 0, s); });
    }
    // im2col of dL/dout ([voxel][co*T + tap'], reading dout at v + off(tap')) serves both gradients:
    //   dW[co][c][T-1-tap'] = sum_v a[v][c] Ad[v][co*T + tap'],   da[v][c] = sum_k Ad[v][k] W[co][c][T-1-tap']
    const int Kp = ((Cin * T + 63) / 64) * 64;
    Tmp Ad = tmp_alloc((size_t)cfg_.max_batch * V0 * Kp * 2 * parts(prec_));
    if (!dry_) {
      void* ad = Ad.ptr; const int mode = (int)prec_;
      add_bwd("head.im2col", [=](cudaStream_t s, int B) { launch_im2col(rt_dout_, ad, B, Cin, R0, k, Kp, mode, s); });
    }
    Act ada; ada.ptr = Ad.ptr; ada.C = Kp; ada.X = ada.Y = ada.Z = R0; ada.B = cfg_.max_batch;
    {
      WgradOut o; o.sm = T; o.sn = -1; o.st = 0; o.ndiv = T; o.sn_hi = (long long)nf * T; o.n_valid = Cin * T;
      emit_wgrad("head.wgrad", act_of(a), ada, 1, 1, G(conv_name + ".weight") + (T - 1), o);
    }
    free_act(a);
    WSrc wd{hw + (T - 1), (long long)T, -1, 0, Cin * T, 0, 0, T, (long long)nf * T};
    GnFuse fh; fh.pname = gn_name; fh.ins = {h}; fh.silu = true; fh.drop_layer = -1;
    GradView da = emit_pointwise("head.dgrad", {ada}, {wd}, nf, R0, nullptr, &fh);
    tmp_free(Ad);
    GradView dx = emit_gn_backward(gn_name, {h}, da, true, -1, nullptr, nullptr, &fh);
    unref(da);
    if (h->grad.valid()) throw std::runtime_error("mdb: head input already has a gradient");
    h->grad = dx;
  });
}

// ------------------------------------------------------------------ time embedding (ddpm_res64.py:132-136, layers.py:680)
void UNet::tape_temb() {
  tape_.push_back([=]() {
    if (dry_) return;
    const int nf = cfg_.nf, tdim = 4 * nf, mb = cfg_.max_batch;
    float* tw0 = P("all_modules.0.weight", {}); float* tb0 = P("all_modules.0.bias", {});
    float* tw1 = P("all_modules.1.weight", {}); float* tb1 = P("all_modules.1.bias", {});
    float* dact = (float*)dmalloc((size_t)mb * tdim * 4);
    float* dt2 = (float*)dmalloc((size_t)mb * tdim * 4);
    float* h1 = (float*)dmalloc((size_t)mb * tdim * 4);
    float* dt1 = (float*)dmalloc((size_t)mb * tdim * 4);
    float* emb = (float*)dmalloc((size_t)mb * nf * 4);
    const float* dd = d_dense_out_; const float* dw = dense_w_; const int dt = dense_total_;
    const long long g_w0 = G("all_modules.0.weight"), g_b0 = G("all_modules.0.bias");
    const long long g_w1 = G("all_modules.1.weight"), g_b1 = G("all_modules.1.bias");
    add_bwd("temb.bwd", [=](cudaStream_t s, int B) {
      launch_dense_bwd_input(dd, dt, dw, dact, B, dt, tdim, s);
      launch_temb_bwd(rt_labels_, tw0, tb0, tw1, tb1, dact, dt2, h1, dt1, emb, B, nf, s);
      launch_outer_sum(dt2, tdim, h1, tdim, rt_grads_ + g_w1, rt_grads_ + g_b1, B, tdim, tdim, rt_accum_ ? 1 : 0, s);
      launch_outer_sum(dt1, tdim, emb, nf, rt_grads_ + g_w0, rt_grads_ + g_b0, B, tdim, nf, rt_accum_ ? 1 : 0, s);
    });
  });
}

}  // namespace mdb

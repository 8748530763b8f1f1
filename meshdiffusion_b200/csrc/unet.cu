// Plan builder + executor for the 3-D DDPM score network. Module numbering follows the reference constructor
// (ddpm_res64.py:57-123 / ddpm_res128.py:59-134) so that checkpoint keys `all_modules.<i>.*` map one-to-one.
#include "unet.h"
#include <algorithm>
#include <cmath>

namespace mdb {

// ------------------------------------------------------------------ arena (first-fit, deterministic)
size_t Arena::alloc(size_t bytes) {
  bytes = (bytes + 1023) & ~size_t(1023);
  for (size_t i = 0; i < blocks_.size(); ++i) {
    if (blocks_[i].free && blocks_[i].size >= bytes) {
      const size_t off = blocks_[i].off;
      if (blocks_[i].size > bytes) {
        Block rest{off + bytes, blocks_[i].size - bytes, true};
        blocks_[i].size = bytes;
        blocks_.insert(blocks_.begin() + i + 1, rest);
      }
      blocks_[i].free = false;
      return off;
    }
  }
  // extend (merging with a trailing free block if there is one)
  if (!blocks_.empty() && blocks_.back().free) {
    blocks_.back().size = bytes;
    blocks_.back().free = false;
    end_ = blocks_.back().off + bytes;
    peak_ = std::max(peak_, end_);
    return blocks_.back().off;
  }
  blocks_.push_back({end_, bytes, false});
  end_ += bytes;
  peak_ = std::max(peak_, end_);
  return blocks_.back().off;
}

void Arena::release(size_t off) {
  for (size_t i = 0; i < blocks_.size(); ++i) {
    if (blocks_[i].off == off && !blocks_[i].free) {
      blocks_[i].free = true;
      if (i + 1 < blocks_.size() && blocks_[i + 1].free) {
        blocks_[i].size += blocks_[i + 1].size;
        blocks_.erase(blocks_.begin() + i + 1);
      }
      if (i > 0 && blocks_[i - 1].free) {
        blocks_[i - 1].size += blocks_[i].size;
        blocks_.erase(blocks_.begin() + i);
      }
      if (!blocks_.empty() && blocks_.back().free) {
        end_ = blocks_.back().off;
        blocks_.pop_back();
      }
      return;
    }
  }
  throw std::runtime_error("mdb: arena release of unknown block");
}

// ------------------------------------------------------------------ UNet plumbing
void* UNet::dmalloc(size_t bytes, bool zero) {
  void* p = nullptr;
  MDB_CUDA_CHECK(cudaMalloc(&p, bytes ? bytes : 16));
  if (zero) MDB_CUDA_CHECK(cudaMemset(p, 0, bytes ? bytes : 16));
  owned_.push_back(p);
  return p;
}

float* UNet::P(const std::string& name, std::vector<long long> shape, float* external) {
  auto it = pindex_.find(name);
  if (it == pindex_.end()) {
    ParamInfo pi;
    pi.name = name; pi.shape = shape; pi.numel = 1;
    for (auto d : shape) pi.numel *= d;
    pi.external = external != nullptr;
    pindex_[name] = (int)params_.size();
    params_.push_back(pi);
    it = pindex_.find(name);
  }
  ParamInfo& pi = params_[it->second];
  if (external) { pi.d = external; pi.external = true; }
  return pi.d;
}

TensP UNet::new_act(int C, int R, bool stats) {
  auto t = std::make_shared<Tens>();
  t->C = C; t->R = R;
  t->bytes = (size_t)cfg_.max_batch * R * R * R * C * esize(prec_) * parts(prec_);
  t->off = arena_.alloc(t->bytes);
  t->ptr = dry_ ? nullptr : arena_base_ + t->off;
  if (stats) {
    const size_t n = (size_t)cfg_.max_batch * C * kStatWords;
    t->stats = dry_ ? nullptr : stats_base_ + stats_cursor_;
    stats_cursor_ += n;
  }
  return t;
}

// Inference: the arena block is recycled as soon as the last forward consumer has been emitted. Training: every
// activation is an input of some backward op, so blocks stay until the owning backward emitter frees them.
void UNet::release(TensP& t) {
  if (train_) return;
  arena_.release(t->off);
  t->live = false;
  t.reset();
}

Act UNet::act_of(const TensP& t) const {
  Act a;
  a.ptr = t->ptr; a.C = t->C; a.X = a.Y = a.Z = t->R; a.B = cfg_.max_batch;
  return a;
}

// Split-K scratch for small problems (few output tiles, long K: the low-resolution levels at small batch). Decided
// from shapes only so the dry sizing pass and the real pass make identical arena allocations.
UNet::Scratch UNet::split_begin(int R, int N, int cin_total, int taps) {
  Scratch s;
  s.S = plan_splits(R, R, R, cfg_.max_batch, N, cin_total, taps, prec_);
  if (s.S > 1) {
    const size_t bytes = (size_t)s.S * cfg_.max_batch * R * R * R * N * sizeof(float);
    s.off = arena_.alloc(bytes);
    s.ptr = dry_ ? nullptr : reinterpret_cast<float*>(arena_base_ + s.off);
    s.active = true;
  }
  return s;
}
void UNet::split_end(Scratch& s) {
  if (s.active) arena_.release(s.off);
  s.active = false;
}

GemmOp* UNet::new_gemm(const std::string& name, bool commit_time) {
  auto g = std::make_unique<GemmOp>();
  g->name = name;
  GemmOp* raw = g.get();
  if (commit_time) commit_gemms_.push_back(std::move(g));
  else gemms_.push_back(std::move(g));
  return raw;
}

// GroupNorm(32, eps 1e-6) + optional SiLU over the channel concatenation of `ins` (torch.cat is never materialised
// in raw form: only this normalised copy, which is the conv's A operand, exists).
TensP UNet::gn(const std::string& pname, const std::vector<TensP>& ins, bool silu, int drop_layer) {
  int C = 0;
  for (auto& t : ins) C += t->C;
  const int R = ins[0]->R;
  float* gamma = P(pname + ".weight", {C});
  float* beta = P(pname + ".bias", {C});
  TensP y = new_act(C, R, false);
  if (dry_) return y;
  NormActArgs na{};
  na.x0 = ins[0]->ptr; na.C0 = ins[0]->C; na.ld0 = ins[0]->C;
  na.x1 = ins.size() > 1 ? ins[1]->ptr : nullptr; na.C1 = ins.size() > 1 ? ins[1]->C : 0; na.ld1 = na.C1;
  na.scale = nullptr; na.shift = nullptr; na.y = y->ptr; na.voxels = (long long)R * R * R; na.silu = silu ? 1 : 0;
  na.tf32 = (int)prec_;
  na.stats0 = ins[0]->stats; na.stats1 = ins.size() > 1 ? ins[1]->stats : nullptr;
  na.gamma = gamma; na.beta = beta; na.groups = 32; na.eps = 1e-6f;
  if (train_ && drop_layer >= 0) {
    add_step("norm_act:" + pname, [na, this, drop_layer](cudaStream_t s, int B) {
      NormActArgs a = na;
      a.drop_thresh = rt_drop_thresh_; a.drop_scale = rt_drop_scale_; a.seed = rt_seed_ + 0x632BE59BD9B4E019ull * (unsigned long long)(drop_layer + 1);
      launch_norm_act(a, B, s);
    });
  } else {
    add_step("norm_act:" + pname, [na](cudaStream_t s, int B) { launch_norm_act(na, B, s); });
  }
  return y;
}

// ResnetBlockDDPM (layers.py:646-689). The NIN shortcut (when in_ch != out_ch) is accumulated into Conv_1's TMEM
// accumulator as extra k-steps over the raw inputs, so the shortcut add is free.
TensP UNet::resblock(const std::vector<TensP>& ins, int out_ch, int midx) {
  const std::string pre = "all_modules." + std::to_string(midx) + ".";
  int Cin = 0;
  for (auto& t : ins) Cin += t->C;
  const int R = ins[0]->R, mb = cfg_.max_batch;
  const int tdim = 4 * cfg_.nf;

  TensP a = gn(pre + "GroupNorm_0", ins, true);
  float* w0 = P(pre + "Conv_0.weight", {out_ch, Cin, 3, 3, 3});
  float* b0 = P(pre + "Conv_0.bias", {out_ch});
  const int doff = dense_cursor_;
  dense_cursor_ += out_ch;
  P(pre + "Dense_0.weight", {out_ch, tdim}, dry_ ? nullptr : dense_w_ + (size_t)doff * tdim);
  P(pre + "Dense_0.bias", {out_ch}, dry_ ? nullptr : dense_b_ + doff);
  if (dry_) { params_[pindex_[pre + "Dense_0.weight"]].external = true; params_[pindex_[pre + "Dense_0.bias"]].external = true; }
  TensP h = new_act(out_ch, R, true);
  Scratch sp0 = split_begin(R, out_ch, Cin, 27);
  if (!dry_) {
    GemmOp* g = new_gemm("res" + std::to_string(midx) + ".conv0");
    g->set_output(prec_, R, R, R, mb, out_ch, h->ptr, out_ch, false);
    g->add_conv({act_of(a)}, w0, 3, 1);
    g->set_bias(b0);
    g->set_rowbias(dense_out_ + doff, dense_total_);
    g->set_stats(h->stats);
    g->enable_splits(sp0.S, sp0.ptr);
    g->finalize(0, false);
    add_step(g->name, [g](cudaStream_t s, int B) { g->launch(s, B); });
  }
  split_end(sp0);
  release(a);
  TensP a2 = gn(pre + "GroupNorm_1", {h}, true, midx);
  release(h);
  float* w1 = P(pre + "Conv_1.weight", {out_ch, out_ch, 3, 3, 3});
  float* b1 = P(pre + "Conv_1.bias", {out_ch});
  float* wn = nullptr; float* bn = nullptr;
  if (Cin != out_ch) {
    wn = P(pre + "NIN_0.W", {Cin, out_ch});
    bn = P(pre + "NIN_0.b", {out_ch});
  } else if (ins.size() != 1) {
    throw std::runtime_error("mdb: identity shortcut over a concatenation is not supported");
  }
  TensP out = new_act(out_ch, R, true);
  Scratch sp1 = split_begin(R, out_ch, out_ch, 27);
  if (!dry_) {
    GemmOp* g = new_gemm("res" + std::to_string(midx) + ".conv1");
    g->set_output(prec_, R, R, R, mb, out_ch, out->ptr, out_ch, false);
    g->add_conv({act_of(a2)}, w1, 3, 1);
    if (wn) {
      std::vector<Act> raw;
      for (auto& t : ins) raw.push_back(act_of(t));
      g->add_pointwise(raw, wn, true);
      float* bsum = (float*)dmalloc(out_ch * 4);
      commit_steps_.push_back({"bias:" + pre, [=](cudaStream_t s, int) { launch_add_vec(b1, bn, bsum, out_ch, s); }});
      g->set_bias(bsum);
    } else {
      g->set_bias(b1);
      g->set_residual(ins[0]->ptr, out_ch, (long long)R * R * R * out_ch, false);
    }
    g->set_stats(out->stats);
    g->enable_splits(sp1.S, sp1.ptr);
    g->finalize(0, false);
    add_step(g->name, [g](cudaStream_t s, int B) { g->launch(s, B); });
  }
  split_end(sp1);
  if (train_) tape_resblock(ins, a, h, a2, out, out_ch, midx, doff);
  release(a2);
  return out;
}

// AttnBlock (layers.py:585-608): single head over all D*H*W positions, head dim = C.
TensP UNet::attn(const TensP& x, int midx) {
  const std::string pre = "all_modules." + std::to_string(midx) + ".";
  const int C = x->C, R = x->R, mb = cfg_.max_batch;
  const int V = R * R * R;
  const int es = esize(prec_);
  TensP hn = gn(pre + "GroupNorm_0", {x}, false);
  float* W[4]; float* Bv[4];
  for (int i = 0; i < 4; ++i) {
    W[i] = P(pre + "NIN_" + std::to_string(i) + ".W", {C, C});
    Bv[i] = P(pre + "NIN_" + std::to_string(i) + ".b", {C});
  }
  TensP qkv = new_act(3 * C, R, false);
  if (!dry_) {
    for (int i = 0; i < 3; ++i) {
      GemmOp* g = new_gemm("attn" + std::to_string(midx) + ".nin" + std::to_string(i));
      g->set_output(prec_, R, R, R, mb, C, (char*)qkv->ptr + (size_t)i * C * es, 3 * C, false);
      g->add_pointwise({act_of(hn)}, W[i], true);
      g->set_bias(Bv[i]);
      g->finalize(0, false);
      add_step(g->name, [g](cudaStream_t s, int B) { g->launch(s, B); });
    }
  }
  release(hn);
  // v^T [B][C][V] so that P.V has a K-major B operand
  TensP vT = new_act(C, R, false);
  if (!dry_) {
    const void* src = qkv->ptr; void* dst = vT->ptr; const int tf = prec_ == kTF32;
    if (prec_ == kBF16X3) {
      // qkv rows are [3C hi | 3C lo]; v^T rows become [V hi | V lo]
      add_step("attn" + std::to_string(midx) + ".vT", [=](cudaStream_t s, int B) {
        launch_transpose_vc(src, 6 * C, 2 * C, dst, B, V, C, 0, s, 2 * V);
        launch_transpose_vc(src, 6 * C, 5 * C, (__nv_bfloat16*)dst + V, B, V, C, 0, s, 2 * V);
      });
    } else
    add_step("attn" + std::to_string(midx) + ".vT", [=](cudaStream_t s, int B) { launch_transpose_vc(src, 3 * C, 2 * C, dst, B, V, C, tf, s); });
  }
  // logits S[b][q][k] in fp32
  auto S = std::make_shared<Tens>();
  S->bytes = (size_t)mb * V * V * 4;
  S->off = arena_.alloc(S->bytes);
  S->ptr = dry_ ? nullptr : arena_base_ + S->off;
  TensP O = new_act(C, R, false);
  if (!dry_) {
    GemmOp* g = new_gemm("attn" + std::to_string(midx) + ".qk");
    g->set_output_strided(prec_, V, 1, 1, mb, V, S->ptr, V, 0, 0, (long long)V * V, true);
    Act q; q.ptr = qkv->ptr; q.C = C; q.ld = 3 * C; q.X = V; q.Y = 1; q.Z = 1; q.B = mb;
    g->add_pointwise({q}, nullptr, true);
    g->set_b_activation((char*)qkv->ptr + (size_t)C * es, C, V, mb, 3 * C, (long long)V * 3 * C);
    g->set_alpha(1.0f / std::sqrt((float)C));
    g->finalize(0, false);
    add_step(g->name, [g](cudaStream_t s, int B) { g->launch(s, B); });
    float* sp = (float*)S->ptr; const int tf = (int)prec_;
    add_step("attn" + std::to_string(midx) + ".softmax", [=](cudaStream_t s, int B) { launch_softmax_rows(sp, (long long)B * V, V, tf, s); });
    GemmOp* g2 = new_gemm("attn" + std::to_string(midx) + ".pv");
    g2->set_output_strided(prec_, V, 1, 1, mb, C, O->ptr, C, 0, 0, (long long)V * C, false);
    Act pa; pa.ptr = S->ptr; pa.C = V; pa.ld = (prec_ == kBF16) ? 2 * V : V; pa.X = V; pa.Y = 1; pa.Z = 1; pa.B = mb;
    g2->add_pointwise({pa}, nullptr, true);
    g2->set_b_activation(vT->ptr, V, C, mb, V, (long long)C * V);
    g2->finalize(0, false);
    add_step(g2->name, [g2](cudaStream_t s, int B) { g2->launch(s, B); });
  }
  if (!train_) arena_.release(S->off);
  { arena_.release(vT->off); vT->live = false; }  // backward multiplies by v itself (K-major there), not by v^T
  release(qkv);
  TensP out = new_act(C, R, true);
  if (!dry_) {
    GemmOp* g = new_gemm("attn" + std::to_string(midx) + ".nin3");
    g->set_output(prec_, R, R, R, mb, C, out->ptr, C, false);
    g->add_pointwise({act_of(O)}, W[3], true);
    g->set_bias(Bv[3]);
    g->set_residual(x->ptr, C, (long long)V * C, false);
    g->set_stats(out->stats);
    g->finalize(0, false);
    add_step(g->name, [g](cudaStream_t s, int B) { g->launch(s, B); });
  }
  if (train_) tape_attn(x, hn, qkv, S, O, out, midx);
  release(O);
  return out;
}

TensP UNet::downsample(const TensP& x, int midx) {
  const std::string pre = "all_modules." + std::to_string(midx) + ".";
  const int C = x->C, R = x->R / 2;
  float* w = P(pre + "Conv_0.weight", {C, C, 3, 3, 3});
  float* b = P(pre + "Conv_0.bias", {C});
  TensP out = new_act(C, R, true);
  Scratch sp = split_begin(R, C, C, 27);
  if (!dry_) {
    GemmOp* g = new_gemm("down" + std::to_string(midx));
    g->set_output(prec_, R, R, R, cfg_.max_batch, C, out->ptr, C, false);
    g->add_conv({act_of(x)}, w, 3, 2);
    g->set_bias(b);
    g->set_stats(out->stats);
    g->enable_splits(sp.S, sp.ptr);
    g->finalize(0, false);
    add_step(g->name, [g](cudaStream_t s, int B) { g->launch(s, B); });
  }
  split_end(sp);
  if (train_) tape_downsample(x, out, midx);
  return out;
}

TensP UNet::upsample(const TensP& x, int midx) {
  const std::string pre = "all_modules." + std::to_string(midx) + ".";
  const int C = x->C, R = x->R * 2;
  float* w = P(pre + "Conv_0.weight", {C, C, 3, 3, 3});
  float* b = P(pre + "Conv_0.bias", {C});
  if (!train_) {
    // Inference: sub-pixel form. Each of the 8 output-parity classes is a 2^3 convolution over the LOW-resolution tensor
    // (8/27 of the FLOPs) writing its strided share of the output; the upsampled tensor never exists. The training plan
    // keeps the materialised form below (its backward differentiates exactly that graph).
    TensP out = new_act(C, R, true);
    if (!dry_) {
      const int r = x->R, mb = cfg_.max_batch;
      float* w8 = (float*)dmalloc((size_t)64 * C * C * sizeof(float));
      commit_steps_.push_back({"upw:" + pre, [=](cudaStream_t s, int) { launch_upconv_weights(w, w8, C, C, s); }});
      const long long es = esize(prec_) * parts(prec_);
      for (int par = 0; par < 8; ++par) {
        const int px = par & 1, py = (par >> 1) & 1, pz = par >> 2;
        GemmOp* g = new_gemm("up" + std::to_string(midx) + ".conv.p" + std::to_string(par));
        char* base = (char*)out->ptr + (((long long)pz * R + py) * R + px) * C * es;
        g->set_output_strided(prec_, r, r, r, mb, C, base, 2LL * C, 2LL * R * C, 2LL * R * R * C, (long long)R * R * R * C, false, C);
        g->add_conv_up2(act_of(x), w8 + (size_t)par * C * C * 8, px, py, pz);
        g->set_bias(b);
        g->set_stats(out->stats);
        g->finalize(0, false);
        add_step(g->name, [g](cudaStream_t s, int B) { g->launch(s, B); });
      }
    }
    return out;
  }
  TensP up = new_act(C, R, false);
  if (!dry_) {
    const void* src = x->ptr; void* dst = up->ptr; const int r = x->R; const int tf = prec_ == kTF32;
    const int Cp = C * parts(prec_);  // X3: a row is 2C bf16 (hi | lo), copied as it is
    add_step("up" + std::to_string(midx) + ".nearest", [=](cudaStream_t s, int B) { launch_upsample2x(src, dst, B, r, r, r, Cp, tf, s); });
  }
  TensP out = new_act(C, R, true);
  Scratch sp = split_begin(R, C, C, 27);
  if (!dry_) {
    GemmOp* g = new_gemm("up" + std::to_string(midx) + ".conv");
    g->set_output(prec_, R, R, R, cfg_.max_batch, C, out->ptr, C, false);
    g->add_conv({act_of(up)}, w, 3, 1);
    g->set_bias(b);
    g->set_stats(out->stats);
    g->enable_splits(sp.S, sp.ptr);
    g->finalize(0, false);
    add_step(g->name, [g](cudaStream_t s, int B) { g->launch(s, B); });
  }
  split_end(sp);
  if (train_) tape_upsample(x, up, out, midx);
  release(up);
  return out;
}

void UNet::build() {
  const int nf = cfg_.nf, R0 = cfg_.image_size, mb = cfg_.max_batch, Cin = cfg_.num_channels;
  const int k = cfg_.stem_ksize, T = k * k * k;
  const int KB = kb_elems(prec_);
  const int tdim = 4 * nf;
  arena_.reset();
  stats_cursor_ = 0;
  dense_cursor_ = 0;
  auto is_attn = [&](int r) { for (int i = 0; i < cfg_.n_attn; ++i) if (cfg_.attn_resolutions[i] == r) return true; return false; };
  auto blocks_at = [&](int lvl) { return (lvl == 0 && cfg_.level0_blocks > 0) ? cfg_.level0_blocks : cfg_.num_res_blocks; };

  int m = 0;
  // --- time embedding MLP (all_modules.0/1)
  float* tw0 = P("all_modules.0.weight", {tdim, nf});
  float* tb0 = P("all_modules.0.bias", {tdim});
  float* tw1 = P("all_modules.1.weight", {tdim, tdim});
  float* tb1 = P("all_modules.1.bias", {tdim});
  m = 2;
  if (!dry_) {
    float* ta = temb_act_; float* dw = dense_w_; float* db = dense_b_; float* dout = dense_out_; const int dt = dense_total_;
    add_step("temb", [=](cudaStream_t s, int B) {
      launch_temb(rt_labels_, tw0, tb0, tw1, tb1, ta, B, nf, s);
      launch_dense(ta, dw, db, dout, B, tdim, dt, s);
    });
  }
  if (train_) tape_temb();
  // --- non-trainable tensors carried by the checkpoint
  float* mask = P("mask", {1, 1, R0, R0, R0});
  if (cfg_.use_pos_bias) P("coords", {1, 3, R0, R0, R0});
  float* posw = P("pos_layer.weight", {nf, 3, k, k, k});
  float* posb = P("pos_layer.bias", {nf});
  float* mw = P("mask_layer.weight", {nf, 1, k, k, k});
  float* mbias = P("mask_layer.bias", {nf});
  (void)posw;
  // --- stem: conv(x) + [pos_layer bias] + mask_layer(mask)   (ddpm_res64.py:148 / ddpm_res128.py:159-162)
  float* sw = P("all_modules.2.weight", {nf, Cin, k, k, k});
  float* sb = P("all_modules.2.bias", {nf});
  m = 3;
  const int Kpad = ((Cin * T + KB - 1) / KB) * KB;
  const int Kpad_m = ((T + KB - 1) / KB) * KB;
  const long long V0 = (long long)R0 * R0 * R0;
  auto A0 = std::make_shared<Tens>();
  A0->bytes = (size_t)mb * V0 * Kpad * esize(prec_) * parts(prec_);
  A0->off = arena_.alloc(A0->bytes);
  A0->ptr = dry_ ? nullptr : arena_base_ + A0->off;
  TensP h0 = new_act(nf, R0, true);
  void* Am = nullptr;
  if (!dry_) {
    // constant field (fp32 [V][nf]) computed once per commit with the same kernels
    float* field = (float*)dmalloc(V0 * nf * 4);
    Am = dmalloc(V0 * Kpad_m * esize(prec_) * parts(prec_));
    float* fbias = (float*)dmalloc(nf * 4);
    const int tf = (int)prec_;
    const bool use_pos = cfg_.use_pos_bias != 0;
    commit_steps_.push_back({"field.bias", [=](cudaStream_t s, int) { launch_add_vec(mbias, use_pos ? posb : nullptr, fbias, nf, s); }});
    commit_steps_.push_back({"field.im2col", [=](cudaStream_t s, int) { launch_im2col(mask, Am, 1, 1, R0, k, Kpad_m, tf, s); }});
    GemmOp* gf = new_gemm("stem.field", true);
    gf->set_output(prec_, R0, R0, R0, 1, nf, field, nf, true);
    Act am; am.ptr = Am; am.C = Kpad_m; am.X = am.Y = am.Z = R0; am.B = 1;
    WSrc wm{mw, (long long)T, 1, 0, T};
    gf->add_pointwise_w({am}, &wm);
    gf->set_bias(fbias);
    gf->finalize(0, false);
    commit_steps_.push_back({"field.gemm", [gf](cudaStream_t s, int) { gf->repack(s); gf->launch(s, 1); }});

    void* a0 = A0->ptr;
    add_step("stem.im2col", [=](cudaStream_t s, int B) { launch_im2col(rt_x_, a0, B, Cin, R0, k, Kpad, tf, s); });
    GemmOp* g = new_gemm("stem.gemm");
    g->set_output(prec_, R0, R0, R0, mb, nf, h0->ptr, nf, false);
    Act a; a.ptr = a0; a.C = Kpad; a.X = a.Y = a.Z = R0; a.B = mb;
    WSrc ws{sw, (long long)Cin * T, 1, 0, Cin * T};
    g->add_pointwise_w({a}, &ws);
    g->set_bias(sb);
    g->set_residual(field, nf, 0, true);
    g->set_stats(h0->stats);
    g->finalize(0, false);
    add_step(g->name, [g](cudaStream_t s, int B) { g->launch(s, B); });
  }
  arena_.release(A0->off);
  if (train_) tape_stem(h0, Am, Kpad, Kpad_m);

  // --- down path
  std::vector<TensP> hs;
  hs.push_back(h0);
  int in_ch = nf;
  for (int lvl = 0; lvl < cfg_.n_levels; ++lvl) {
    const int res = R0 >> lvl;
    for (int b = 0; b < blocks_at(lvl); ++b) {
      const int out_ch = nf * cfg_.ch_mult[lvl];
      TensP h = resblock({hs.back()}, out_ch, m++);
      in_ch = out_ch;
      if (is_attn(res)) {
        TensP h2 = attn(h, m++);
        release(h);
        h = h2;
      }
      hs.push_back(h);
    }
    if (lvl != cfg_.n_levels - 1) hs.push_back(downsample(hs.back(), m++));
  }
  // --- middle
  TensP h;
  {
    TensP h1 = resblock({hs.back()}, in_ch, m++);
    TensP h2 = attn(h1, m++);
    release(h1);
    h = resblock({h2}, in_ch, m++);
    release(h2);
  }
  // --- up path
  for (int lvl = cfg_.n_levels - 1; lvl >= 0; --lvl) {
    const int res = R0 >> lvl;
    for (int b = 0; b < blocks_at(lvl) + 1; ++b) {
      const int out_ch = nf * cfg_.ch_mult[lvl];
      TensP skip = hs.back();
      hs.pop_back();
      TensP hn = resblock({h, skip}, out_ch, m++);
      release(h);
      release(skip);
      h = hn;
    }
    if (is_attn(res)) {
      TensP h2 = attn(h, m++);
      release(h);
      h = h2;
    }
    if (lvl != 0) {
      TensP u = upsample(h, m++);
      release(h);
      h = u;
    }
  }
  if (!hs.empty()) throw std::runtime_error("mdb: skip stack not empty");
  // --- head: GroupNorm -> SiLU -> conv(nf -> channels)
  const std::string head_gn = "all_modules." + std::to_string(m);
  TensP a = gn("all_modules." + std::to_string(m++), {h}, true);
  TensP head_in = h;
  release(h);
  float* hw = P("all_modules." + std::to_string(m) + ".weight", {Cin, nf, k, k, k});
  float* hb = P("all_modules." + std::to_string(m) + ".bias", {Cin});
  ++m;
  // The head has only `Cin` (= 4) output channels: as an implicit GEMM it would stream all 27/125 shifted A tiles for
  // an N=4 product. Instead: (1) ONE unshifted GEMM projects every voxel onto all taps at once,
  //   P[v][tap*Cout + co] = sum_c a[v][c] * W[co][c][tap]      (N = taps*Cout = 108 / 500, K = nf),
  // (2) a bandwidth kernel gathers out[v][co] = bias[co] + sum_tap P[v + off(tap)][tap*Cout + co].
  if (Cin == 4) {
    const int Np = ((T * Cin + 7) / 8) * 8;
    const bool pf32 = prec_ != kBF16;  // tf32 / split bf16: the per-tap projections stay fp32
    auto Pt = std::make_shared<Tens>();
    Pt->bytes = (size_t)mb * V0 * Np * (pf32 ? 4 : 2);
    Pt->off = arena_.alloc(Pt->bytes);
    Pt->ptr = dry_ ? nullptr : arena_base_ + Pt->off;
    if (!dry_) {
      GemmOp* g = new_gemm("head.proj");
      g->set_output(prec_, R0, R0, R0, mb, T * Cin, Pt->ptr, Np, pf32);
      WSrc ws{hw, (long long)nf * T, (long long)T, 0, nf, Cin, 1};
      g->add_pointwise_w({act_of(a)}, &ws);
      g->finalize(0, false);
      add_step(g->name, [g](cudaStream_t s, int B) { g->launch(s, B); });
      const void* pp = Pt->ptr;
      add_step("head.shift_sum", [=](cudaStream_t s, int B) { launch_tap_shift_sum(pp, Np, pf32 ? 1 : 0, hb, rt_out_, B, R0, k, Cin, s); });
    }
    arena_.release(Pt->off);
  } else if (!dry_) {
    GemmOp* g = new_gemm("head.conv");
    g->set_output_strided(prec_, R0, R0, R0, mb, Cin, nullptr, 1, R0, (long long)R0 * R0, (long long)Cin * V0, true);
    g->set_out_col_stride(V0);
    g->add_conv({act_of(a)}, hw, k, 1);
    g->set_bias(hb);
    g->finalize(0, false);
    add_step(g->name, [g, this](cudaStream_t s, int B) { g->launch(s, B, rt_out_); });
  }
  if (train_) tape_head(head_in, a, head_gn, "all_modules." + std::to_string(m - 1));
  release(a);
  dense_total_ = dense_cursor_;
  stats_doubles_ = stats_cursor_;
  if (train_) {
    // emit the backward plan: the emitters recorded during the forward pass, in reverse order
    bwd_count_ = 0;
    for (auto it = tape_.rbegin(); it != tape_.rend(); ++it) {
      touched_.clear();
      (*it)();
      // every gradient this emitter writes is final once all of its launches have run (the dry pass counts the same
      // launches, so a GPU-less plan answers mdb_unet_grad_ready too)
      for (auto& n : touched_) grad_ready_[n] = bwd_count_;
    }
    tape_.clear();
    if (arena_.in_use() != 0) throw std::runtime_error("mdb: training plan leaked " + std::to_string(arena_.in_use()) + " arena bytes");
  }
}

UNet::UNet(const UNetConfig& cfg, bool dry_only) : cfg_(cfg), prec_(precision_from_int(cfg.precision)) {
  if (cfg_.image_size % (1 << (cfg_.n_levels - 1)) != 0) throw std::runtime_error("mdb: image_size not divisible by 2^(levels-1)");
  if (cfg_.nf % 32 != 0) throw std::runtime_error("mdb: nf must be a multiple of 32 (GroupNorm(32))");
  train_ = cfg_.training != 0;
  if (const char* e = getenv("MDB_GRAPH_MAX_BATCH")) graph_max_batch_ = atoi(e);  // 0 disables graph replay
  if (train_ && prec_ == kTF32) throw std::runtime_error("mdb: the training plan is built for bf16 or bf16x3 operands");
  dry_ = true;
  build();
  // allocate everything the dry run sized
  arena_bytes_ = arena_.peak();
  {
    long long off = 0;
    for (auto& p : params_) { goff_[p.name] = off; off += p.numel; }
  }
  if (dry_only) return;
  arena_base_ = (char*)dmalloc(arena_bytes_, false);
  stats_base_ = (long long*)dmalloc(stats_doubles_ * sizeof(long long));
  const int tdim = 4 * cfg_.nf;
  temb_act_ = (float*)dmalloc((size_t)cfg_.max_batch * tdim * 4);
  dense_w_ = (float*)dmalloc((size_t)dense_total_ * tdim * 4);
  dense_b_ = (float*)dmalloc((size_t)dense_total_ * 4);
  dense_out_ = (float*)dmalloc((size_t)cfg_.max_batch * dense_total_ * 4);
  if (train_) d_dense_out_ = (float*)dmalloc((size_t)cfg_.max_batch * dense_total_ * 4);
  for (auto& p : params_)
    if (!p.external) p.d = (float*)dmalloc(p.numel * 4);
  dry_ = false;
  build();
  for (auto& g : gemms_) flops_ += g->flops;
  for (auto& g : bwd_gemms_) bwd_flops_ += g->flops;
  for (auto& g : wgrads_) bwd_flops_ += g->flops;
  MDB_CUDA_CHECK(cudaDeviceSynchronize());
}

UNet::~UNet() {
  drop_graphs();
  if (capture_stream_) cudaStreamDestroy(capture_stream_);
  gemms_.clear();
  bwd_gemms_.clear();
  wgrads_.clear();
  commit_gemms_.clear();
  for (void* p : owned_) cudaFree(p);
}

void UNet::set_param(const std::string& name, const float* src, long long numel, bool dev, cudaStream_t s) {
  auto it = pindex_.find(name);
  if (it == pindex_.end()) throw std::runtime_error("mdb: unknown parameter " + name);
  ParamInfo& p = params_[it->second];
  if (p.numel != numel) throw std::runtime_error("mdb: parameter " + name + " expects " + std::to_string(p.numel) + " elements, got " + std::to_string(numel));
  MDB_CUDA_CHECK(cudaMemcpyAsync(p.d, src, numel * 4, dev ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, s));
  committed_ = false;
}

void UNet::get_param(const std::string& name, float* dst, long long numel, bool dev, cudaStream_t s) {
  auto it = pindex_.find(name);
  if (it == pindex_.end()) throw std::runtime_error("mdb: unknown parameter " + name);
  ParamInfo& p = params_[it->second];
  if (p.numel != numel) throw std::runtime_error("mdb: parameter " + name + " size mismatch");
  MDB_CUDA_CHECK(cudaMemcpyAsync(dst, p.d, numel * 4, dev ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, s));
  MDB_CUDA_CHECK(cudaStreamSynchronize(s));
}

void UNet::commit(cudaStream_t s) {
  drop_graphs();  // packed weights are rewritten in place, but derived pointers are only guaranteed per commit
  for (auto& st : commit_steps_) st.fn(s, 1);
  for (auto& g : gemms_) g->repack(s);
  for (auto& g : bwd_gemms_) g->repack(s);
  MDB_CUDA_CHECK(cudaStreamSynchronize(s));
  committed_ = true;
}

void UNet::drop_graphs() {
  for (auto& g : graphs_) if (g.exec) cudaGraphExecDestroy(g.exec);
  graphs_.clear();
}

void UNet::forward(const float* x, const float* labels, float* out, int B, cudaStream_t s, bool allow_graph) {
  if (!committed_) throw std::runtime_error("mdb: parameters changed, call commit() before forward()");
  if (B < 1 || B > cfg_.max_batch) throw std::runtime_error("mdb: batch out of range");
  rt_x_ = x; rt_labels_ = labels; rt_out_ = out;
  if (allow_graph && !train_ && B <= graph_max_batch_) {
    FwdGraph* fg = nullptr;
    for (auto& g : graphs_) if (g.x == x && g.labels == labels && g.out == out && g.B == B) fg = &g;
    if (!fg) {
      if (graphs_.size() >= 8) drop_graphs();
      graphs_.push_back({x, labels, out, B, 0, nullptr});
      fg = &graphs_.back();
    }
    if (fg->exec) { MDB_CUDA_CHECK(cudaGraphLaunch(fg->exec, s)); return; }
    if (fg->uses++ >= 1) {
      // second call with these buffers: capture (the first ran eagerly, so every kernel attribute is configured)
      if (!capture_stream_) MDB_CUDA_CHECK(cudaStreamCreateWithFlags(&capture_stream_, cudaStreamNonBlocking));
      cudaGraph_t graph = nullptr;
      MDB_CUDA_CHECK(cudaStreamBeginCapture(capture_stream_, cudaStreamCaptureModeThreadLocal));
      try {
        MDB_CUDA_CHECK(cudaMemsetAsync(stats_base_, 0, stats_doubles_ * sizeof(long long), capture_stream_));
        for (auto& st : steps_) st.fn(capture_stream_, B);
      } catch (...) {
        cudaStreamEndCapture(capture_stream_, &graph);
        if (graph) cudaGraphDestroy(graph);
        throw;
      }
      MDB_CUDA_CHECK(cudaStreamEndCapture(capture_stream_, &graph));
      cudaError_t e = cudaGraphInstantiate(&fg->exec, graph, 0);
      cudaGraphDestroy(graph);
      if (e != cudaSuccess) { fg->exec = nullptr; MDB_CUDA_CHECK(e); }
      MDB_CUDA_CHECK(cudaGraphLaunch(fg->exec, s));
      return;
    }
  }
  MDB_CUDA_CHECK(cudaMemsetAsync(stats_base_, 0, stats_doubles_ * sizeof(long long), s));
  for (auto& st : steps_) st.fn(s, B);
}

std::vector<std::pair<std::string, float>> UNet::profile(const float* x, const float* labels, float* out, int B, cudaStream_t s) {
  if (!committed_) throw std::runtime_error("mdb: commit() first");
  rt_x_ = x; rt_labels_ = labels; rt_out_ = out;
  std::vector<std::pair<std::string, float>> res;
  std::vector<cudaEvent_t> ev(steps_.size() + 1);
  for (auto& e : ev) MDB_CUDA_CHECK(cudaEventCreate(&e));
  MDB_CUDA_CHECK(cudaMemsetAsync(stats_base_, 0, stats_doubles_ * sizeof(long long), s));
  MDB_CUDA_CHECK(cudaEventRecord(ev[0], s));
  for (size_t i = 0; i < steps_.size(); ++i) {
    steps_[i].fn(s, B);
    MDB_CUDA_CHECK(cudaEventRecord(ev[i + 1], s));
  }
  MDB_CUDA_CHECK(cudaStreamSynchronize(s));
  for (size_t i = 0; i < steps_.size(); ++i) {
    float ms = 0;
    MDB_CUDA_CHECK(cudaEventElapsedTime(&ms, ev[i], ev[i + 1]));
    res.push_back({steps_[i].name, ms});
  }
  for (auto& e : ev) cudaEventDestroy(e);
  return res;
}

}  // namespace mdb

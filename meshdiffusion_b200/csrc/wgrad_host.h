// Host-side construction of tcgen05 weight-gradient operations (see wgrad_tc.cuh).
#pragma once
#include <map>
#include "gemm_host.h"
#include "wgrad_tc.cuh"

namespace mdb {

// Where G[tap][m][n] goes: out[m*sm + n*sn + tap*st], or with ndiv: n -> (n / ndiv, n % ndiv) with strides (sn_hi, sn).
struct WgradOut {
  float* ptr = nullptr;
  long long sm = 0, sn = 0, st = 0;
  int ndiv = 0;
  long long sn_hi = 0;
  int m_valid = 0, n_valid = 0;  // rows / columns actually written (0 = all channels of the operands)
};

// SMs the split-K plan is sized for. A constant (not the device query) so that the GPU-less sizing pass and the real
// pass agree on every scratch size.
constexpr int kPlanSMs = 148;

struct WgradPlan {
  int m_tiles = 0, n_tiles = 0, n_groups = 0, taps = 0, max_splits = 1;
  bool halo = false, flat = false;
  Geometry geo{};
  size_t scratch_bytes = 0;
};
// dY extents (X,Y,Z,B) = output positions of the forward op; M = dY channels, N = X-operand channels.
WgradPlan plan_wgrad(int X, int Y, int Z, int B, int M, int N, int ksize, int stride);

class WgradOp {
 public:
  std::string name;
  double flops = 0;
  // dy: [B][Z][Y][X][M] (C = M), x: the forward op's input activation (C = N; for stride 2 at twice the extents).
  // ksize 1 (pointwise; any stride-1 geometry, positions are flattened) or 3 (stride 1 pad 1, or stride 2 pad-high).
  // x3: both operands are split-bf16 tensors ((hi, lo) rows of logical pitch ld, gemm_host.h::kBF16X3)
  void init(const Act& dy, const Act& x, int ksize, int stride, const WgradOut& out, float* scratch, bool x3 = false);
  // accumulate: out += G instead of out = G (micro-batch gradient accumulation)
  void launch(cudaStream_t s, int B, bool accumulate, float* out_ptr = nullptr);
  const WgradPlan& plan() const { return plan_; }

 private:
  WgradPlan plan_;
  WgradParams base_{};
  Act dy_, x_;
  int ksize_ = 1, stride_ = 1, M_ = 0, N_ = 0;
  bool x3_ = false;
  WgradOut out_;
  std::map<int, WgradParams> cache_;  // tensor maps encoded for a given runtime batch
  const WgradParams& params_for(int B);
};

struct WgradReduceArgs {
  const float* partial; int splits, taps, Mp, Np, M, N;
  float* out; long long sm, sn, st; int ndiv; long long sn_hi; int accumulate;
};
void launch_wgrad_reduce(const WgradReduceArgs& a, cudaStream_t s);

}  // namespace mdb

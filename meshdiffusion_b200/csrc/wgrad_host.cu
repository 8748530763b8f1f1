// Host-side builders for the tcgen05 weight-gradient kernel (see wgrad_tc.cuh) and its split-K reduction.
#define MDB_WGRAD_KERNEL_IMPL
#include "wgrad_host.h"
#include <cstdlib>

namespace mdb {

WgradPlan plan_wgrad(int X, int Y, int Z, int B, int M, int N, int ksize, int stride) {
  WgradPlan pl;
  if (ksize != 1 && ksize != 3) throw std::runtime_error("mdb: wgrad supports 1x1x1 and 3x3x3 kernels");
  pl.flat = ksize == 1;
  long long tiles;
  if (pl.flat) {
    pl.geo = {128, 1, 1, 1};
    pl.n_groups = 1; pl.taps = 1;
    tiles = ((long long)B * X * Y * Z + 127) / 128;
  } else {
    pl.geo = pick_geometry(X, Y, Z);
    pl.halo = stride == 1 && pl.geo.bz == 1 && pl.geo.bb == 1 && pl.geo.bx % 8 == 0 &&
              pl.geo.bx * (pl.geo.by + 2) <= kWgXRowsMax && Y >= pl.geo.by;
    pl.n_groups = pl.halo ? 9 : 27;
    pl.taps = 27;
    tiles = 1LL * ((X + pl.geo.bx - 1) / pl.geo.bx) * ((Y + pl.geo.by - 1) / pl.geo.by) * ((Z + pl.geo.bz - 1) / pl.geo.bz) *
            ((B + pl.geo.bb - 1) / pl.geo.bb);
  }
  pl.m_tiles = (M + 127) / 128;
  pl.n_tiles = (N + 127) / 128;
  const long long items = 1LL * pl.m_tiles * pl.n_tiles * pl.n_groups;
  long long S = kPlanSMs / items;
  if (S < 1) S = 1;
  if (S > tiles) S = tiles;
  pl.max_splits = (int)S;
  pl.scratch_bytes = (size_t)S * pl.taps * pl.m_tiles * 128 * pl.n_tiles * 128 * sizeof(float);
  return pl;
}

void WgradOp::init(const Act& dy, const Act& x, int ksize, int stride, const WgradOut& out, float* scratch, bool x3) {
  dy_ = dy; x_ = x; ksize_ = ksize; stride_ = stride; out_ = out; x3_ = x3;
  M_ = dy.C; N_ = x.C;
  plan_ = plan_wgrad(dy.X, dy.Y, dy.Z, dy.B, M_, N_, ksize, stride);
  if (ksize == 3 && stride == 1 && (x.X != dy.X || x.Y != dy.Y || x.Z != dy.Z)) throw std::runtime_error("mdb: wgrad extent mismatch");
  if (ksize == 3 && stride == 2 && (x.X != 2 * dy.X || x.Y != 2 * dy.Y || x.Z != 2 * dy.Z)) throw std::runtime_error("mdb: stride-2 wgrad extent mismatch");
  if (ksize == 1 && x.voxels() != dy.voxels()) throw std::runtime_error("mdb: pointwise wgrad extent mismatch");
  WgradParams& p = base_;
  p.bx = plan_.geo.bx; p.by = plan_.geo.by; p.bz = plan_.geo.bz; p.bb = plan_.geo.bb;
  p.m_tiles = plan_.m_tiles; p.n_tiles = plan_.n_tiles;
  p.taps = plan_.taps;
  p.Mp = plan_.m_tiles * 128; p.Np = plan_.n_tiles * 128;
  p.partial = scratch;
  p.y_lo = x3 ? (int)dy.row() : 0;
  p.x_lo = x3 ? (int)x.row() : 0;
  { const char* f = getenv("MDB_WG_DBG"); p.dbg = f ? atoi(f) : 0; }
  p.n_groups = plan_.n_groups;
  const int xrows = plan_.halo ? p.bx * (p.by + 2) : 128;
  p.x_chunk_bytes = xrows * kRowBytes;
  p.tap_shift16 = plan_.halo ? (p.bx * kRowBytes) >> 4 : 0;
  int g = 0;
  if (plan_.flat) {
    p.groups[g++] = WgradGroup{0, 0, 0, 0, 1, {0, 0, 0}};
  } else if (plan_.halo) {
    for (int kz = 0; kz < 3; ++kz)
      for (int kx = 0; kx < 3; ++kx) {
        WgradGroup gr{0, (int8_t)(kx - 1), -1, (int8_t)(kz - 1), 3, {0, 0, 0}};
        for (int ky = 0; ky < 3; ++ky) gr.tap[ky] = (int8_t)((kz * 3 + ky) * 3 + kx);
        p.groups[g++] = gr;
      }
  } else {
    for (int kz = 0; kz < 3; ++kz)
      for (int ky = 0; ky < 3; ++ky)
        for (int kx = 0; kx < 3; ++kx) {
          const int8_t tap = (int8_t)((kz * 3 + ky) * 3 + kx);
          if (stride == 1) p.groups[g++] = WgradGroup{0, (int8_t)(kx - 1), (int8_t)(ky - 1), (int8_t)(kz - 1), 1, {tap, 0, 0}};
          else p.groups[g++] = WgradGroup{(int8_t)((kx & 1) | ((ky & 1) << 1) | ((kz & 1) << 2)), (int8_t)(kx >> 1), (int8_t)(ky >> 1), (int8_t)(kz >> 1), 1, {tap, 0, 0}};
        }
  }
  flops = 2.0 * dy.voxels() * dy.B * (double)M_ * N_ * plan_.taps;  // algorithmic (X3 issues 3x the MMAs)
}

const WgradParams& WgradOp::params_for(int B) {
  auto it = cache_.find(B);
  if (it != cache_.end()) return it->second;
  WgradParams p = base_;
  const long long es = 2;
  // X3: a row is [ld hi | ld lo]; the map's channel extent reaches from the view's first hi channel to its last lo one
  const long long pp = x3_ ? 2 : 1;
  auto cdim = [&](const Act& a) { return (uint64_t)(x3_ ? a.row() + a.C : a.C); };
  uint64_t dims[5], strides[4];
  uint32_t box[5];
  if (plan_.flat) {
    const long long rows = (long long)B * dy_.voxels();
    p.tx = (int)((rows + 127) / 128); p.ty = p.tz = p.tb = 1;
    auto enc = [&](CUtensorMap* m, const Act& a) {
      dims[0] = cdim(a); dims[1] = rows; dims[2] = dims[3] = dims[4] = 1;
      strides[0] = pp * a.row() * es; strides[1] = strides[0] * rows; strides[2] = strides[1]; strides[3] = strides[1];
      box[0] = 64; box[1] = 128; box[2] = box[3] = box[4] = 1;
      encode_map(m, kBF16, 5, a.ptr, dims, strides, box);
    };
    enc(&p.ymap, dy_);
    enc(&p.xmap[0], x_);
  } else {
    p.tx = (dy_.X + p.bx - 1) / p.bx; p.ty = (dy_.Y + p.by - 1) / p.by; p.tz = (dy_.Z + p.bz - 1) / p.bz;
    p.tb = (B + p.bb - 1) / p.bb;
    auto enc = [&](CUtensorMap* m, const Act& a, int halo, int sub, int px, int py, int pz) {
      char* base = static_cast<char*>(a.ptr);
      const long long sx = pp * a.row() * es, sy = sx * a.X, sz = sy * a.Y, sb = sz * a.Z;
      dims[0] = cdim(a); dims[4] = B;
      if (sub == 1) {
        dims[1] = a.X; dims[2] = a.Y; dims[3] = a.Z;
        strides[0] = sx; strides[1] = sy; strides[2] = sz; strides[3] = sb;
      } else {
        dims[1] = (a.X - px + sub - 1) / sub; dims[2] = (a.Y - py + sub - 1) / sub; dims[3] = (a.Z - pz + sub - 1) / sub;
        strides[0] = sx * sub; strides[1] = sy * sub; strides[2] = sz * sub; strides[3] = sb;
        base += px * sx + py * sy + pz * sz;
      }
      box[0] = 64; box[1] = p.bx; box[2] = p.by + halo; box[3] = p.bz; box[4] = p.bb;
      encode_map(m, kBF16, 5, base, dims, strides, box);
    };
    enc(&p.ymap, dy_, 0, 1, 0, 0, 0);
    if (stride_ == 1) {
      enc(&p.xmap[0], x_, plan_.halo ? 2 : 0, 1, 0, 0, 0);
    } else {
      for (int par = 0; par < 8; ++par) enc(&p.xmap[par], x_, 0, 2, par & 1, (par >> 1) & 1, (par >> 2) & 1);
    }
  }
  const long long tiles = 1LL * p.tx * p.ty * p.tz * p.tb;
  const long long items = 1LL * p.m_tiles * p.n_tiles * p.n_groups;
  long long S = kPlanSMs / items;
  if (S < 1) S = 1;
  if (S > tiles) S = tiles;
  if (S > plan_.max_splits) S = plan_.max_splits;
  p.splits = (int)S;
  return cache_.emplace(B, p).first->second;
}

// ------------------------------------------------------------------ split reduction + scatter to the parameter layout
// One thread per (tap, m, n): the split partials of that element are summed in split order (deterministic) and the
// result goes to its slot of the parameter layout. (A thread per (m, n) looping over the taps left 16 K threads with
// 432 dependent loads each: 38 us per launch, 5.6 ms per backward pass.)
__global__ void __launch_bounds__(256) wgrad_reduce_kernel(WgradReduceArgs a) {
  const long long per_tap = (long long)a.M * a.N;
  const long long total = per_tap * a.taps;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int t = (int)(i / per_tap);
    const long long r = i - (long long)t * per_tap;
    const int m = (int)(r / a.N), n = (int)(r % a.N);
    float acc = 0.f;
    for (int s = 0; s < a.splits; ++s) acc += __ldg(a.partial + (((long long)s * a.taps + t) * a.Mp + m) * a.Np + n);
    const long long noff = a.ndiv ? (long long)(n % a.ndiv) * a.sn + (long long)(n / a.ndiv) * a.sn_hi : (long long)n * a.sn;
    float* o = a.out + m * a.sm + noff + t * a.st;
    *o = a.accumulate ? *o + acc : acc;
  }
}

void launch_wgrad_reduce(const WgradReduceArgs& a, cudaStream_t s) {
  const long long total = (long long)a.M * a.N * a.taps;
  long long blocks = (total + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  wgrad_reduce_kernel<<<(unsigned)blocks, 256, 0, s>>>(a);
  MDB_CUDA_CHECK(cudaGetLastError());
}

void WgradOp::launch(cudaStream_t s, int B, bool accumulate, float* out_ptr) {
  if (B < 1 || B > dy_.B) throw std::runtime_error("mdb: wgrad batch out of range");
  const WgradParams& p = params_for(B);
  static bool configured_dev[64] = {};  // the attribute is per device
  int dev = 0;
  MDB_CUDA_CHECK(cudaGetDevice(&dev));
  bool& configured = configured_dev[dev < 64 ? dev : 63];
  if (!configured || dev >= 63) {
    MDB_CUDA_CHECK(cudaFuncSetAttribute(wgrad_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kWgSmemBytes));
    MDB_CUDA_CHECK(cudaFuncSetAttribute(wgrad_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kWgSmemBytes));
    configured = true;
  }
  const int grid = p.m_tiles * p.n_tiles * p.n_groups * p.splits;
  if (x3_) wgrad_tc_kernel<true><<<grid, kWgThreads, kWgSmemBytes, s>>>(p);
  else wgrad_tc_kernel<false><<<grid, kWgThreads, kWgSmemBytes, s>>>(p);
  MDB_CUDA_CHECK(cudaGetLastError());
  WgradReduceArgs r{};
  r.partial = p.partial; r.splits = p.splits; r.taps = p.taps; r.Mp = p.Mp; r.Np = p.Np; r.M = out_.m_valid ? out_.m_valid : M_; r.N = out_.n_valid ? out_.n_valid : N_;
  r.out = out_ptr ? out_ptr : out_.ptr; r.sm = out_.sm; r.sn = out_.sn; r.st = out_.st; r.ndiv = out_.ndiv; r.sn_hi = out_.sn_hi;
  r.accumulate = accumulate ? 1 : 0;
  launch_wgrad_reduce(r, s);
}

}  // namespace mdb

// Host-side builders for the tcgen05 implicit-GEMM kernel (see gemm_tc.cuh).
#include "gemm_host.h"
#include "elementwise.cuh"
#include <cstring>
#include <cstdlib>
#include <mutex>

namespace mdb {

// ------------------------------------------------------------------ driver entry point (no libcuda link dependency)
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode() {
  static PFN_encodeTiled fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q);
    if (e != cudaSuccess || q != cudaDriverEntryPointSuccess || !f)
      throw std::runtime_error("mdb: cuTensorMapEncodeTiled not available (needs an sm_90+ driver)");
    fn = reinterpret_cast<PFN_encodeTiled>(f);
  });
  return fn;
}

void encode_map(CUtensorMap* m, Precision prec, int rank, void* base, const uint64_t* dims,
                const uint64_t* strides_bytes /*rank-1*/, const uint32_t* box) {
  cuuint64_t gd[5], gs[4];
  cuuint32_t bd[5], es[5];
  for (int i = 0; i < rank; ++i) { gd[i] = dims[i]; bd[i] = box[i]; es[i] = 1; }
  for (int i = 0; i + 1 < rank; ++i) gs[i] = strides_bytes[i];
  CUtensorMapDataType dt = prec == kTF32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  CUresult r = get_encode()(m, dt, rank, base, gd, gs, bd, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                            CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    std::string msg = "mdb: cuTensorMapEncodeTiled failed (" + std::to_string((int)r) + ") rank " +
                      std::to_string(rank) + " dims";
    for (int i = 0; i < rank; ++i) msg += " " + std::to_string(dims[i]);
    msg += " box";
    for (int i = 0; i < rank; ++i) msg += " " + std::to_string(box[i]);
    throw std::runtime_error(msg);
  }
}

static int sm_count_or_default() {
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) {
    cudaGetLastError();
    return 148;
  }
  return n;
}

int sm_count() {
  static int n = 0;
  if (!n) {
    int dev = 0;
    MDB_CUDA_CHECK(cudaGetDevice(&dev));
    MDB_CUDA_CHECK(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev));
  }
  return n;
}

Geometry pick_geometry(int X, int Y, int Z) {
  if (Y == 1 && Z == 1) return {128, 1, 1, 1};
  int bx = X < 8 ? X : 8;
  int by = 128 / bx;
  if (by > 16) by = 16;
  if (by > Y) by = Y;
  int rem = 128 / (bx * by);
  int bz = rem < Z ? rem : Z;
  int bb = rem / bz;
  return {bx, by, bz, bb};
}

int plan_splits(int X, int Y, int Z, int B, int N, int cin_total, int taps, Precision prec) {
  const Geometry g = pick_geometry(X, Y, Z);
  const int tiles_m = ((X + g.bx - 1) / g.bx) * ((Y + g.by - 1) / g.by) * ((Z + g.bz - 1) / g.bz) * ((B + g.bb - 1) / g.bb);
  const int block_n = N <= 32 ? 32 : 128;
  const int tiles = tiles_m * ((N + block_n - 1) / block_n);
  const int ksteps = ((cin_total + kb_elems(prec) - 1) / kb_elems(prec)) * taps * (prec == kBF16X3 ? 3 : 1);
  if (tiles > 49 || ksteps < 48) return 1;
  int S = 148 / tiles;
  if (S > 16) S = 16;
  if (S > ksteps / 8) S = ksteps / 8;
  return S < 2 ? 1 : S;
}

void GemmOp::enable_splits(int S, float* scratch) {
  if (S <= 1) return;
  if (pair || p.ocs != 1 || p.out_fp32 || p.bias_on_m || p.alpha != 1.f || p.res_fp32)
    throw std::runtime_error("mdb: split-K is only wired for plain NDHWC conv outputs");
  if (p.osx != (long long)p.N * parts(prec) || (p.res && p.rsx != (long long)p.N * parts(prec)))
    throw std::runtime_error("mdb: split-K needs dense [B][V][N] output / residual");
  splits = S;
  p.splits = S;
  p.partial = scratch;
  p.split_stride = (long long)p.Bn * p.X * p.Y * p.Z * p.N;
}

GemmOp::~GemmOp() {
  if (d_loads) cudaFree(d_loads);
  if (d_ks0) cudaFree(d_ks0);
  if (d_wpacked && owns_w) cudaFree(d_wpacked);
}

void GemmOp::set_output_strided(Precision pr, int X, int Y, int Z, int B, int N, void* out, long long osx,
                                long long osy, long long osz, long long osb, bool out_fp32, long long lo_off) {
  prec = pr;
  geo = pick_geometry(X, Y, Z);
  if (geo.bx * geo.by * geo.bz * geo.bb != kBlockM) throw std::runtime_error("mdb: unsupported tile geometry");
  if (geo.bb > 1 && (geo.bx * geo.by * geo.bz) % 32 != 0)
    throw std::runtime_error("mdb: multi-sample tiles need a multiple of 32 rows per sample");
  if (geo.bb > 4) throw std::runtime_error("mdb: at most 4 samples per tile");
  p.bx = geo.bx; p.by = geo.by; p.bz = geo.bz; p.bb = geo.bb;
  p.X = X; p.Y = Y; p.Z = Z; p.Bn = B;
  p.tx = (X + geo.bx - 1) / geo.bx; p.ty = (Y + geo.by - 1) / geo.by;
  p.tz = (Z + geo.bz - 1) / geo.bz; p.tb = (B + geo.bb - 1) / geo.bb;
  p.N = N;
  block_n = N <= 32 ? 32 : 128;
  p.n_tiles_n = (N + block_n - 1) / block_n;
  { const char* f = getenv("MDB_DBG_FLAGS"); p.dbg_flags = f ? atoi(f) : 0; }
  {
    // CTA pairs (tcgen05 cta_group::2) whenever there are enough M-tiles to keep all 74 pairs busy
    const char* e = getenv("MDB_CTA_PAIRS");
    const int tiles_m = p.tx * p.ty * p.tz * p.tb;
    pair = block_n == 128 && tiles_m * p.n_tiles_n >= 2 * (sm_count_or_default() / 2) && !(e && e[0] == '0');
  }
  p.out = out;
  p.osx = osx; p.osy = osy; p.osz = osz; p.osb = osb;
  p.out_fp32 = out_fp32 ? 1 : 0;
  p.out_lo_off = 0;
  if (prec == kBF16X3 && !out_fp32) {  // (hi, lo) rows: physical pitch 2x the logical one, lo parts one logical row behind
    p.out_lo_off = lo_off >= 0 ? lo_off : osx;
    p.osx *= 2; p.osy *= 2; p.osz *= 2; p.osb *= 2;
  }
  {
    // TF32 operands: tensor cores truncate fp32 inputs to 10 mantissa bits; rounding the stored activations to
    // nearest instead removes that systematic bias (measured on the full res64 net: rel-L2 vs fp32 2.5e-3 -> 1.5e-3,
    // on par with stock cuDNN/cuBLAS TF32). MDB_TF32_ROUND_STORE=0 restores plain fp32 stores.
    const char* e = getenv("MDB_TF32_ROUND_STORE");
    p.round_out = (prec == kTF32 && !out_fp32 && !(e && e[0] == '0')) ? 1 : 0;
  }
  p.alpha = 1.f;
  p.ocs = 1;
  p.kb_elems = kb_elems(prec);
}

void GemmOp::set_output(Precision pr, int X, int Y, int Z, int B, int N, void* out, long long ldc, bool out_fp32) {
  set_output_strided(pr, X, Y, Z, B, N, out, ldc, ldc * X, ldc * X * Y, ldc * X * Y * Z, out_fp32);
}

int GemmOp::add_amap(const Act& a, int halo, int sub, int px, int py, int pz, int part) {
  if (n_amaps >= kMaxAMaps) throw std::runtime_error("mdb: too many A tensor maps");
  if (halo > 0 && (geo.bz != 1 || geo.bb != 1)) throw std::runtime_error("mdb: halo needs a (bx,by,1,1) tile");
  const long long es = esize(prec);
  const long long prow = a.row() * parts(prec);  // physical row pitch in elements
  uint64_t dims[5], strides[4];
  uint32_t box[5];
  char* base = static_cast<char*>(a.ptr) + (long long)part * a.row() * es;
  if (sub == 1) {
    dims[0] = a.C; dims[1] = a.X; dims[2] = a.Y; dims[3] = a.Z; dims[4] = a.B;
    strides[0] = prow * es; strides[1] = strides[0] * a.X; strides[2] = strides[1] * a.Y; strides[3] = strides[2] * a.Z;
  } else {
    dims[0] = a.C; dims[1] = (a.X - px + sub - 1) / sub; dims[2] = (a.Y - py + sub - 1) / sub;
    dims[3] = (a.Z - pz + sub - 1) / sub; dims[4] = a.B;
    const long long sx = prow * es, sy = sx * a.X, sz = sy * a.Y, sb = sz * a.Z;
    strides[0] = sx * sub; strides[1] = sy * sub; strides[2] = sz * sub; strides[3] = sb;
    base += px * sx + py * sy + pz * sz;
  }
  box[0] = kb_elems(prec); box[1] = geo.bx; box[2] = geo.by + halo; box[3] = geo.bz; box[4] = geo.bb;
  encode_map(&p.amap[n_amaps], prec, 5, base, dims, strides, box);
  return n_amaps++;
}

void GemmOp::add_load_x(int tm_hi, int tm_lo, int nk, int rows, int jrows, int dx, int dy, int dz, int c0, int wsrc,
                        int wc0, int tap0, int tapj) {
  if (prec != kBF16X3) { add_load(tm_hi, nk, rows, jrows, dx, dy, dz, c0, wsrc, wc0, tap0, tapj, 0); return; }
  if (pair) {
    // CTA pairs: a (hi, lo) couple of stages -- (A hi, W hi) then (A lo, W lo) -- from which the MMA warp forms the three
    // products itself (GemmSeg::x3pair): every operand byte crosses L2 -> SMEM once
    add_load(tm_hi, nk, rows, jrows, dx, dy, dz, c0, wsrc, wc0, tap0, tapj, 0);
    add_load(tm_lo, nk, rows, jrows, dx, dy, dz, c0, wsrc, wc0, tap0, tapj, 1);
    return;
  }
  // K-extension form (single CTAs: small problems, split-K). Small terms first: (A lo, W hi) and (A hi, W lo) are ~2^-9
  // of the leading product
  add_load(tm_lo, nk, rows, jrows, dx, dy, dz, c0, wsrc, wc0, tap0, tapj, 0);
  add_load(tm_hi, nk, rows, jrows, dx, dy, dz, c0, wsrc, wc0, tap0, tapj, 1);
  add_load(tm_hi, nk, rows, jrows, dx, dy, dz, c0, wsrc, wc0, tap0, tapj, 0);
}

void GemmOp::add_load(int tmap, int nk, int rows, int jrows, int dx, int dy, int dz, int c0, int wsrc, int wc0,
                      int tap0, int tapj, int wpart) {
  if ((int)loads.size() >= kMaxLoads) throw std::runtime_error("mdb: load table overflow");
  if (rows > kAStageRows) throw std::runtime_error("mdb: A box exceeds the stage size");
  LoadEntry e{};
  e.tmap = (uint8_t)tmap; e.nk = (uint8_t)nk; e.rows = (uint8_t)rows; e.jrows = (uint8_t)jrows;
  e.dx = (int8_t)dx; e.dy = (int8_t)dy; e.dz = (int8_t)dz; e.wsrc = (uint8_t)wsrc;
  e.c0 = (uint16_t)c0; e.wc0 = (uint16_t)wc0; e.tap0 = (uint8_t)tap0; e.tapj = (uint8_t)tapj; e.wpart = (uint16_t)wpart;
  loads.push_back(e);
  ksteps += nk;
}

void GemmOp::add_conv(const std::vector<Act>& srcs, const float* w, int k, int stride) {
  int ctot = 0;
  for (auto& s : srcs) ctot += s.C;
  const int T = k * k * k;
  add_conv_w(srcs, WSrc{w, 1LL * ctot * T, (long long)T, 1, ctot}, k, stride);
}

// Data gradient of a stride-1 k^3 convolution = the same convolution over dY with the weight transposed (Cout <-> Cin)
// and every tap mirrored: W'[ci][co][tap] = W[co][ci][T-1-tap].
void GemmOp::add_conv_dgrad(const Act& dy, const float* w_oidhw, int cin_total, int k) {
  const int T = k * k * k;
  add_conv_w({dy}, WSrc{w_oidhw + (T - 1), (long long)T, 1LL * cin_total * T, -1, dy.C}, k, 1);
}

void GemmOp::add_conv_w(const std::vector<Act>& srcs, const WSrc& wsrc, int k, int stride) {
  const int KB = kb_elems(prec);
  int ctot = 0;
  for (auto& s : srcs) ctot += s.C;
  const int T = k * k * k;
  const int ws = add_wsrc(wsrc);
  const int pad = k / 2;
  flops += 2.0 * p.X * p.Y * p.Z * p.Bn * (double)p.N * ctot * T;
  int coff = 0;
  if (stride == 1) {
    const bool reuse = geo.bz == 1 && geo.bb == 1 && geo.bx * (geo.by + k - 1) <= kAStageRows && p.Y >= geo.by;
    const bool x3 = prec == kBF16X3;
    for (auto& s : srcs) {
      const int tm = add_amap(s, reuse ? k - 1 : 0);
      const int tl = x3 ? add_amap(s, reuse ? k - 1 : 0, 1, 0, 0, 0, 1) : tm;
      for (int c0 = 0; c0 < s.C; c0 += KB) {
        if (reuse) {
          for (int dz = 0; dz < k; ++dz)
            for (int dx = 0; dx < k; ++dx)
              add_load_x(tm, tl, k, geo.bx * (geo.by + k - 1), geo.bx, dx - pad, -pad, dz - pad, c0, ws, coff + c0,
                         (dz * k) * k + dx, k);
        } else {
          for (int dz = 0; dz < k; ++dz)
            for (int dy = 0; dy < k; ++dy)
              for (int dx = 0; dx < k; ++dx)
                add_load_x(tm, tl, 1, kBlockM, 0, dx - pad, dy - pad, dz - pad, c0, ws, coff + c0, (dz * k + dy) * k + dx, 0);
        }
      }
      coff += s.C;
    }
  } else if (stride == 2) {
    // layers.py:626-643: pad one voxel on the high side only, then stride-2 VALID conv: in = 2*o + d.
    // Tap d reads the parity-(d&1) sub-grid at coordinate o + (d>>1); coordinate == sub-grid size -> zero fill = pad.
    if (k != 3) throw std::runtime_error("mdb: stride-2 conv supports k=3 only");
    const bool x3 = prec == kBF16X3;
    for (auto& s : srcs) {
      int tm[8], tl[8];
      for (int par = 0; par < 8; ++par) tm[par] = add_amap(s, 0, 2, par & 1, (par >> 1) & 1, (par >> 2) & 1);
      for (int par = 0; par < 8; ++par) tl[par] = x3 ? add_amap(s, 0, 2, par & 1, (par >> 1) & 1, (par >> 2) & 1, 1) : tm[par];
      for (int c0 = 0; c0 < s.C; c0 += KB)
        for (int dz = 0; dz < 3; ++dz)
          for (int dy = 0; dy < 3; ++dy)
            for (int dx = 0; dx < 3; ++dx) {
              const int par = (dx & 1) | ((dy & 1) << 1) | ((dz & 1) << 2);
              add_load_x(tm[par], tl[par], 1, kBlockM, 0, dx >> 1, dy >> 1, dz >> 1, c0, ws, coff + c0, (dz * 3 + dy) * 3 + dx, 0);
            }
      coff += s.C;
    }
  } else {
    throw std::runtime_error("mdb: unsupported stride");
  }
}

void GemmOp::add_conv_up2(const Act& s, const float* w8, int px, int py, int pz) {
  const int KB = kb_elems(prec);
  const int ws = add_wsrc(WSrc{w8, 8LL * s.C, 8, 1, s.C});
  flops += 2.0 * p.X * p.Y * p.Z * p.Bn * (double)p.N * s.C * 8;
  const bool x3 = prec == kBF16X3;
  // effective tap e in {0,1} of an axis with output parity q reads the input at offset e - 1 + q
  const bool reuse = geo.bz == 1 && geo.bb == 1 && geo.bx * (geo.by + 1) <= kAStageRows && p.Y >= geo.by;
  const int tm = add_amap(s, reuse ? 1 : 0);
  const int tl = x3 ? add_amap(s, reuse ? 1 : 0, 1, 0, 0, 0, 1) : tm;
  for (int c0 = 0; c0 < s.C; c0 += KB) {
    for (int ez = 0; ez < 2; ++ez)
      for (int ex = 0; ex < 2; ++ex) {
        if (reuse) {  // the two y-taps share one box with a 1-row halo
          add_load_x(tm, tl, 2, geo.bx * (geo.by + 1), geo.bx, ex - 1 + px, -1 + py, ez - 1 + pz, c0, ws, c0, (ez * 2) * 2 + ex, 2);
        } else {
          for (int ey = 0; ey < 2; ++ey)
            add_load_x(tm, tl, 1, kBlockM, 0, ex - 1 + px, ey - 1 + py, ez - 1 + pz, c0, ws, c0, (ez * 2 + ey) * 2 + ex, 0);
        }
      }
  }
}

void GemmOp::add_pointwise(const std::vector<Act>& srcs, const float* w, bool w_in_out) {
  int ctot = 0;
  for (auto& s : srcs) ctot += s.C;
  if (!w) { add_pointwise_w(srcs, nullptr); return; }
  WSrc ws = w_in_out ? WSrc{w, 1, (long long)p.N, 0, ctot} : WSrc{w, (long long)ctot, 1, 0, ctot};
  add_pointwise_w(srcs, &ws);
}

void GemmOp::add_pointwise_w(const std::vector<Act>& srcs, const WSrc* w) {
  const int KB = kb_elems(prec);
  int ctot = 0;
  for (auto& s : srcs) ctot += s.C;
  int ws = 0;
  if (w) ws = add_wsrc(*w);
  flops += 2.0 * p.X * p.Y * p.Z * p.Bn * (double)p.N * ctot;
  int coff = 0;
  for (auto& s : srcs) {
    const int tm = add_amap(s, 0);
    const int tl = prec == kBF16X3 ? add_amap(s, 0, 1, 0, 0, 0, 1) : tm;
    for (int c0 = 0; c0 < s.C; c0 += KB) add_load_x(tm, tl, 1, kBlockM, 0, 0, 0, 0, c0, ws, coff + c0, 0, 0);
    coff += s.C;
  }
}

void GemmOp::set_residual(const void* res, long long ldr, long long batch_stride, bool fp32) {
  p.res = res;
  p.batch_fastest = batch_stride == 0 ? 1 : 0;  // a residual shared by every sample: keep its slice L2-resident
  p.rsx = ldr; p.rsy = ldr * p.X; p.rsz = ldr * p.X * p.Y; p.rsb = batch_stride;
  p.res_fp32 = fp32 ? 1 : 0;
  p.res_lo_off = 0;
  if (prec == kBF16X3 && !fp32) {
    p.res_lo_off = ldr;
    p.rsx *= 2; p.rsy *= 2; p.rsz *= 2; p.rsb *= 2;
  }
}

void GemmOp::set_gn_backward(const void* x0, long long ld0, int c0, const void* x1, long long ld1, const void* consts, int silu,
                             float* part) {
  if (prec == kTF32 || p.out_fp32 || p.ocs != 1) throw std::runtime_error("mdb: the GroupNorm-backward epilogue is built for bf16 / bf16x3 NDHWC outputs");
  if (p.N % 32 != 0 || (x1 && c0 % 32 != 0)) throw std::runtime_error("mdb: GroupNorm-backward epilogue needs 32-channel aligned sources");
  if (splits > 1) throw std::runtime_error("mdb: GroupNorm-backward epilogue cannot be combined with split-K");
  gnb = true;
  // X3: the GroupNorm inputs are (hi, lo) rows -- physical pitches twice the logical ones, lo parts one logical row behind
  const long long pp = parts(prec);
  p.res = x0; p.res_fp32 = 0; p.batch_fastest = 0;
  p.rsx = pp * ld0; p.rsy = p.rsx * p.X; p.rsz = p.rsy * p.Y; p.rsb = p.rsz * p.Z;
  p.res1 = x1; p.res_c0 = x1 ? c0 : p.N;
  p.r1sx = pp * ld1; p.r1sy = p.r1sx * p.X; p.r1sz = p.r1sy * p.Y; p.r1sb = p.r1sz * p.Z;
  p.res_lo_off = prec == kBF16X3 ? ld0 : 0;
  p.res1_lo_off = prec == kBF16X3 ? ld1 : 0;
  p.gnb_c = reinterpret_cast<const float4*>(consts);
  p.gnb_silu = silu;
  p.gnb_part = part;
}

void GemmOp::encode_bmap(void* ptr, int K, int N, int batch, long long rsb, long long bsb) {
  uint64_t dims[3] = {(uint64_t)K, (uint64_t)N, (uint64_t)batch};
  uint64_t strides[2] = {(uint64_t)rsb, (uint64_t)bsb};
  uint32_t box[3] = {(uint32_t)kb_elems(prec), (uint32_t)(pair ? block_n / 2 : block_n), 1};
  encode_map(&p.bmap, prec, 3, ptr, dims, strides, box);
}

void GemmOp::set_b_activation(void* ptr, int K, int N, int batch, long long rs, long long bs) {
  b_from_act = true;
  p.b_batched = 1;
  const long long es = esize(prec);
  if (prec == kBF16X3) {
    // rows are (hi, lo) pairs: the lo parts are addressed as K coordinates [rs, rs + K) of the same map
    if (K % kb_elems(prec) != 0) throw std::runtime_error("mdb: X3 activation-B operands need K to be a multiple of 64");
    b_lo_off = rs;
    encode_bmap(ptr, (int)(rs + K), N, batch, 2 * rs * es, 2 * bs * es);
    return;
  }
  encode_bmap(ptr, K, N, batch, rs * es, bs * es);
}

// ------------------------------------------------------------------ weight packing (device gather)
struct PackWSrc { const float* ptr; long long sn, sc, st; int cvalid; int ndiv; long long sn_hi; int cdiv; long long sc_hi; };
struct PackArgs { PackWSrc w[4]; };

__device__ __forceinline__ float round_tf32(float x) {
  uint32_t u;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(x));
  return __uint_as_float(u);
}

// MODE: 0 = bf16, 1 = tf32 (rna), 2 = split bf16 (entry.wpart selects hi = bf16(w) or lo = bf16(w - hi)).
// One thread = 8 consecutive K elements (one 16- / 32-byte store) of EVERY k-step of one load entry for one output row: the
// entry / source / offset arithmetic is done once per 8 * nk outputs. (The first version, one thread per packed element with
// two 64-bit divisions and a table walk each, made the per-optimiser-step re-pack of the training engine instruction-bound:
// 6-8 ms for 2.9 GB of traffic.)
template <int MODE>
__global__ void __launch_bounds__(256) pack_weights_kernel(const LoadEntry* __restrict__ loads, const int* __restrict__ load_ks0,
                                                         int n_loads, const __grid_constant__ PackArgs args, int N, int ksteps,
                                                         int KB, void* __restrict__ out) {
  const int vpk = KB >> 3;  // 8-element vectors per k-step
  const long long total = 1LL * N * n_loads * vpk;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int v8 = (int)(idx % vpk);
    const long long t = idx / vpk;
    const int l = (int)(t % n_loads);
    const int n = (int)(t / n_loads);
    const LoadEntry e = loads[l];
    const PackWSrc& w = args.w[e.wsrc];
    const long long noff = w.ndiv ? (long long)(n % w.ndiv) * w.sn + (long long)(n / w.ndiv) * w.sn_hi : (long long)n * w.sn;
    const int c0 = e.wc0 + v8 * 8;
    long long coff[8];  // (may be negative: mirrored sources point at their last tap and walk backwards)
    unsigned valid = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int c = c0 + i;
      if (c < w.cvalid) valid |= 1u << i;
      coff[i] = noff + (w.cdiv ? (long long)(c % w.cdiv) * w.sc + (long long)(c / w.cdiv) * w.sc_hi : (long long)c * w.sc);
    }
    const long long obase = ((long long)n * ksteps + load_ks0[l]) * KB + v8 * 8;
    for (int j = 0; j < e.nk; ++j) {
      const long long toff = (long long)(e.tap0 + j * e.tapj) * w.st;
      float v[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) v[i] = (valid >> i) & 1u ? __ldg(w.ptr + coff[i] + toff) : 0.f;
      const long long o = obase + (long long)j * KB;
      if (MODE == 1) {
        float4* op = reinterpret_cast<float4*>(reinterpret_cast<float*>(out) + o);
        op[0] = make_float4(round_tf32(v[0]), round_tf32(v[1]), round_tf32(v[2]), round_tf32(v[3]));
        op[1] = make_float4(round_tf32(v[4]), round_tf32(v[5]), round_tf32(v[6]), round_tf32(v[7]));
      } else {
        uint4 pk;
        __nv_bfloat16* h = reinterpret_cast<__nv_bfloat16*>(&pk);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const __nv_bfloat16 hi = __float2bfloat16(v[i]);
          h[i] = (MODE == 2 && e.wpart) ? __float2bfloat16(v[i] - __bfloat162float(hi)) : hi;
        }
        *reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(out) + o) = pk;
      }
    }
  }
}

void GemmOp::repack(cudaStream_t stream) {
  if (b_from_act) return;
  if (!d_ks0) {  // first k-step of every load entry: built once, reused by every re-pack
    std::vector<int> ks0;
    int run = 0;
    for (size_t l = 0; l < loads.size(); ++l) { ks0.push_back(run); run += loads[l].nk; }
    if (run != ksteps) throw std::runtime_error("mdb: load table does not cover the packed K extent");
    MDB_CUDA_CHECK(cudaMalloc(&d_ks0, ks0.size() * sizeof(int)));
    MDB_CUDA_CHECK(cudaMemcpy(d_ks0, ks0.data(), ks0.size() * sizeof(int), cudaMemcpyHostToDevice));
  }
  if (wsrcs.size() > 4) throw std::runtime_error("mdb: too many weight sources");
  PackArgs args{};
  for (size_t i = 0; i < wsrcs.size(); ++i) args.w[i] = {wsrcs[i].ptr, wsrcs[i].sn, wsrcs[i].sc, wsrcs[i].st, wsrcs[i].cvalid, wsrcs[i].ndiv, wsrcs[i].sn_hi, wsrcs[i].cdiv, wsrcs[i].sc_hi};
  const int KB = kb_elems(prec), n_loads = (int)loads.size();
  const long long total = 1LL * p.N * n_loads * (KB / 8);
  int blocks = (int)((total + 255) / 256);
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (prec == kTF32)
    pack_weights_kernel<1><<<blocks, 256, 0, stream>>>(d_loads, d_ks0, n_loads, args, p.N, ksteps, KB, d_wpacked);
  else if (prec == kBF16X3)
    pack_weights_kernel<2><<<blocks, 256, 0, stream>>>(d_loads, d_ks0, n_loads, args, p.N, ksteps, KB, d_wpacked);
  else
    pack_weights_kernel<0><<<blocks, 256, 0, stream>>>(d_loads, d_ks0, n_loads, args, p.N, ksteps, KB, d_wpacked);
  MDB_CUDA_CHECK(cudaGetLastError());
}

void GemmOp::finalize(cudaStream_t stream, bool pack) {
  if (loads.empty()) throw std::runtime_error("mdb: GemmOp without loads");
  p.b_explicit_k = 0;
  if (b_from_act && prec == kBF16X3) {
    // activation-B operand in the split layout: every entry names the K coordinate of its B tile itself
    // ((A hi, B hi), (A hi, B lo), (A lo, B hi) cannot be a running column of one matrix)
    for (auto& e : loads) {
      const long long k0 = (long long)e.wc0 + (e.wpart ? b_lo_off : 0);
      if (k0 > 65535) throw std::runtime_error("mdb: X3 activation-B K coordinate exceeds the table's 16 bits");
      e.wc0 = (uint16_t)k0;
    }
    p.b_explicit_k = 1;
  }
  MDB_CUDA_CHECK(cudaMalloc(&d_loads, loads.size() * sizeof(LoadEntry)));
  MDB_CUDA_CHECK(cudaMemcpyAsync(d_loads, loads.data(), loads.size() * sizeof(LoadEntry), cudaMemcpyHostToDevice, stream));
  p.loads = d_loads;
  p.n_loads = (int)loads.size();
  if (p.splits < 1) p.splits = 1;
  // pipeline segments: runs of identical entries; plain (nk == 1) entries are paired two per stage. The stage size is the
  // largest group of this op and the ring takes as many stages as fit in the 227 KB next to the epilogue scratch.
  {
    const int btile = block_n * kRowBytes / (pair ? 2 : 1);
    const int max_stage = pair ? (2 * 128 * kRowBytes + 2 * 64 * kRowBytes) : (kAStageBytes + 3 * 128 * kRowBytes);
    const bool x3pair = pair && prec == kBF16X3;
    {
      // two M-tiles per CTA (weight tiles shared by both): bf16 / tf32 pair kernels with packed weights and enough tiles to
      // fill every pair with 4-tile work items; MDB_M2=0 switches it off
      const char* e = getenv("MDB_M2");
      const int tiles_m = p.tx * p.ty * p.tz * p.tb;
      m2 = pair && prec != kBF16X3 && !b_from_act && block_n == 128 && !(e && e[0] == '0') &&
           (long long)tiles_m * p.n_tiles_n >= 4LL * (sm_count_or_default() / 2);
    }
    stage_need = 0;
    p.n_segs = 0;
    auto push = [&](int n_groups, int epg, const LoadEntry& e, int couple) {
      if (n_groups <= 0) return;
      if (p.n_segs >= kMaxSegs) throw std::runtime_error("mdb: too many pipeline segments");
      GemmSeg sg{};
      sg.n_groups = n_groups; sg.epg = epg; sg.nk = e.nk;
      sg.a_bytes = e.rows * kRowBytes;
      sg.a_stride = (sg.a_bytes + 1023) / 1024 * 1024;
      sg.jbytes = e.jrows * kRowBytes;
      sg.x3pair = couple;
      const int need = m2 ? 2 * sg.a_stride + e.nk * btile : epg * (sg.a_stride + e.nk * btile);
      if (need > (m2 ? kMaxDynSmem / 2 : max_stage)) throw std::runtime_error("mdb: pipeline group exceeds the stage size");
      if (need > stage_need) stage_need = need;
      p.segs[p.n_segs++] = sg;
      p.total_groups += n_groups;
    };
    p.total_groups = 0;
    size_t i = 0;
    while (i < loads.size()) {
      size_t j = i;
      while (j < loads.size() && loads[j].nk == loads[i].nk && loads[j].rows == loads[i].rows && loads[j].jrows == loads[i].jrows) ++j;
      const int run = (int)(j - i);
      if (x3pair) {
        if (run % 2 != 0) throw std::runtime_error("mdb: X3 stage couples need an even run of entries");
        push(run, 1, loads[i], 1);
      } else if (m2) {
        push(run, 1, loads[i], 0);  // one entry per group: its box for both sub-tiles + the shared weight tiles
      } else if (loads[i].nk == 1 && 2 * (loads[i].rows * kRowBytes + btile) <= max_stage) {
        push(run / 2, 2, loads[i], 0);
        push(run % 2, 1, loads[i], 0);
      } else {
        push(run, 1, loads[i], 0);
      }
      i = j;
    }
  }
  if (p.splits > p.total_groups) { p.splits = p.total_groups; splits = p.splits; }
  if (!b_from_act) {
    const long long ktot = 1LL * ksteps * kb_elems(prec);
    const long long bytes = ktot * p.N * esize(prec);
    MDB_CUDA_CHECK(cudaMalloc(&d_wpacked, bytes));
    owns_w = true;
    p.b_batched = 0;
    encode_bmap(d_wpacked, (int)ktot, p.N, 1, ktot * esize(prec), bytes);
    if (pack) repack(stream);
  }
  MDB_CUDA_CHECK(cudaStreamSynchronize(stream));
}

template <int BN, bool TF32, bool CG2, bool GNB = false, bool X3 = false, bool M2 = false>
static void launch_impl(const GemmParams& p, int grid, cudaStream_t stream) {
  static bool configured[64] = {};  // the attribute is per device
  auto kern = gemm_tc_kernel<BN, TF32, CG2, GNB, X3, M2>;
  const int smem = GemmCfg<BN, CG2>::kFixedBytes + p.n_stages * p.stage_bytes;
  int dev = 0;
  MDB_CUDA_CHECK(cudaGetDevice(&dev));
  if (dev >= 64 || !configured[dev]) {
    MDB_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxDynSmem));
    if (dev < 64) configured[dev] = true;
  }
  if (CG2) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(kGemmThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = 1;
    MDB_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kern, p));
  } else {
    kern<<<grid, kGemmThreads, smem, stream>>>(p);
  }
  MDB_CUDA_CHECK(cudaGetLastError());
}

void GemmOp::launch(cudaStream_t stream, int B, void* out_override) const {
  GemmParams p = this->p;
  {
    // operand ring of this op: stage = its largest pipeline group, as many stages as the 227 KB allow
    const int fixed = 1024 + 24 * block_n * 4 + (2 * kMaxStages + 4) * 8 + 16;  // GemmCfg<block_n, *>::kFixedBytes
    p.stage_bytes = (stage_need + 1023) / 1024 * 1024;
    int ns = (kMaxDynSmem - fixed) / p.stage_bytes;
    // measured (profiles/r02_bench_stages_4_vs_5.txt): a fifth 42 KB stage fits for the halo convolutions but is 1-2 %
    // SLOWER in all three operand modes than four -- the feed is bounded by L2 -> SMEM bytes per MMA, not by bytes in flight
    int cap = 4;
    if (const char* e = getenv("MDB_MAX_STAGES")) { const int c = atoi(e); if (c >= 2) cap = c; }
    if (ns > cap) ns = cap;
    p.n_stages = ns > kMaxStages ? kMaxStages : ns;
    if (p.n_stages < 2) throw std::runtime_error("mdb: operand ring needs at least two stages");
  }
  if (B > 0) {
    if (B > this->p.Bn) throw std::runtime_error("mdb: batch exceeds the batch the op was built for");
    p.Bn = B;
    p.tb = (B + p.bb - 1) / p.bb;
  }
  if (out_override) p.out = out_override;
  const int tiles_m = p.tx * p.ty * p.tz * p.tb;
  const bool tf = prec == kTF32;
  const bool x3 = prec == kBF16X3;
  if (gnb) {
    if (tf || p.splits > 1) throw std::runtime_error("mdb: GroupNorm-backward epilogue: bf16 / bf16x3, no split-K");
    p.gnb_drop_thresh = rt_drop_thresh; p.gnb_drop_scale = rt_drop_scale; p.gnb_seed = rt_seed;
    if (x3) {  // (m2 is never chosen for X3)
      if (pair) {
        const int pairs = sm_count() / 2, work = (tiles_m + 1) / 2 * p.n_tiles_n;
        launch_impl<128, false, true, true, true>(p, 2 * (work < pairs ? work : pairs), stream);
      } else {
        const int total = tiles_m * p.n_tiles_n;
        const int grid = total < sm_count() ? total : sm_count();
        if (block_n == 32) launch_impl<32, false, false, true, true>(p, grid, stream); else launch_impl<128, false, false, true, true>(p, grid, stream);
      }
      return;
    }
    if (pair) {
      const int work = (m2 ? (tiles_m + 3) / 4 : (tiles_m + 1) / 2) * p.n_tiles_n;
      const int pairs = sm_count() / 2;
      if (m2) launch_impl<128, false, true, true, false, true>(p, 2 * (work < pairs ? work : pairs), stream);
      else launch_impl<128, false, true, true>(p, 2 * (work < pairs ? work : pairs), stream);
    } else {
      const int total = tiles_m * p.n_tiles_n;
      const int grid = total < sm_count() ? total : sm_count();
      if (block_n == 32) launch_impl<32, false, false, true>(p, grid, stream); else launch_impl<128, false, false, true>(p, grid, stream);
    }
    return;
  }
  if (pair) {
    const int work = (m2 ? (tiles_m + 3) / 4 : (tiles_m + 1) / 2) * p.n_tiles_n;
    const int pairs = sm_count() / 2;
    const int grid = 2 * (work < pairs ? work : pairs);
    if (m2) { if (tf) launch_impl<128, true, true, false, false, true>(p, grid, stream); else launch_impl<128, false, true, false, false, true>(p, grid, stream); }
    else if (tf) launch_impl<128, true, true>(p, grid, stream);
    else if (x3) launch_impl<128, false, true, false, true>(p, grid, stream);
    else launch_impl<128, false, true>(p, grid, stream);
    return;
  }
  const int total = tiles_m * p.n_tiles_n * (p.splits > 1 ? p.splits : 1);
  int grid = total < sm_count() ? total : sm_count();
  if (block_n == 32) {
    if (tf) launch_impl<32, true, false>(p, grid, stream);
    else if (x3) launch_impl<32, false, false, false, true>(p, grid, stream);
    else launch_impl<32, false, false>(p, grid, stream);
  } else {
    if (tf) launch_impl<128, true, false>(p, grid, stream);
    else if (x3) launch_impl<128, false, false, false, true>(p, grid, stream);
    else launch_impl<128, false, false>(p, grid, stream);
  }
  if (p.splits > 1) {
    SplitReduceArgs a{};
    a.partial = p.partial; a.split_stride = p.split_stride; a.splits = p.splits;
    a.bias = p.bias; a.rowbias = p.rowbias; a.rowbias_ld = p.rowbias_ld;
    a.res = p.res; a.res_batch_stride = p.rsb;
    a.out = p.out; a.stats = p.stats; a.voxels = (long long)p.X * p.Y * p.Z; a.N = p.N; a.tf32 = tf ? 1 : (x3 ? 2 : 0);
    if (x3) a.res_batch_stride = p.rsb / 2;  // the reduction kernel takes logical strides
    launch_split_reduce(a, p.Bn, stream);
  }
}

}  // namespace mdb

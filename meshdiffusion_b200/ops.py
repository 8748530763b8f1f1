"""Operator-level wrappers over the C ABI (used by the parity tests; the engine itself stays inside the library).

Activations are NDHWC torch tensors on the GPU: bfloat16 for precision='bf16', float32 for precision='tf32', and for
precision='bf16x3' (split bf16) bfloat16 rows of 2C entries: the hi parts bf16(v) of the C channels followed by their
lo parts bf16(v - hi).
"""
import ctypes

import torch

from . import _native

PRECISIONS = {"bf16": 0, "tf32": 1, "bf16x3": 2}
STAT_WORDS = 4  # csrc/gn_stats.cuh: (sum lo, sum hi, sumsq lo, sumsq hi); value = lo * 2^-24 + hi * 2^16


def stats_to_words(stats):
    """float64 [B,C,2] (sum, sum of squares) -> the library's int64 [B,C,4] split fixed-point record."""
    v = stats.double()
    hi = torch.round(v / 65536.0)
    lo = torch.round((v - hi * 65536.0) * 16777216.0)
    return torch.stack([lo[..., 0], hi[..., 0], lo[..., 1], hi[..., 1]], dim=-1).to(torch.int64).contiguous()


def words_to_stats(words):
    w = words.double()
    return torch.stack([w[..., 0] / 16777216.0 + w[..., 1] * 65536.0, w[..., 2] / 16777216.0 + w[..., 3] * 65536.0], dim=-1)


def _act_dtype(precision):
    return torch.float32 if precision == "tf32" else torch.bfloat16


def to_ndhwc(x_ncdhw, precision):
    """[B,C,D,H,W] fp32 -> contiguous [B,D,H,W,C] in the operand dtype ([B,D,H,W,2C] = hi | lo for 'bf16x3')."""
    y = x_ncdhw.permute(0, 2, 3, 4, 1).contiguous()
    if precision == "bf16x3":
        hi = y.to(torch.bfloat16)
        lo = (y.float() - hi.float()).to(torch.bfloat16)
        return torch.cat([hi, lo], dim=-1).contiguous()
    return y.to(_act_dtype(precision))


def from_ndhwc(y, precision=None):
    if precision == "bf16x3":
        C = y.shape[-1] // 2
        y = y[..., :C].float() + y[..., C:].float()
    return y.float().permute(0, 4, 1, 2, 3).contiguous()


def conv3d(x, weight, bias=None, stride=1, rowbias=None, residual=None, want_stats=False, precision="bf16"):
    """nn.Conv3d (k in {1,3,5}; stride 1 'same' or the Downsample stride-2 pad-high variant) on NDHWC input.

    x: [B,Z,Y,X,Cin]; weight: fp32 [Cout,Cin,k,k,k]. Returns y [B,Zo,Yo,Xo,Cout] (and stats [B,Cout,2] float64).
    """
    L = _native.lib()
    assert x.is_cuda and x.is_contiguous() and x.dtype == _act_dtype(precision)
    B, Z, Y, X, Cin = x.shape
    parts = 2 if precision == "bf16x3" else 1
    Cin //= parts
    Cout, k = weight.shape[0], weight.shape[2]
    assert weight.shape[1] == Cin
    w = weight.detach().float().contiguous()
    y = torch.empty((B, Z // stride, Y // stride, X // stride, Cout * parts), device=x.device, dtype=x.dtype)
    stats = torch.zeros((B, Cout, STAT_WORDS), device=x.device, dtype=torch.int64) if want_stats else None
    b = bias.detach().float().contiguous() if bias is not None else None
    rb = rowbias.detach().float().contiguous() if rowbias is not None else None
    if residual is not None:
        assert residual.shape == y.shape and residual.dtype == y.dtype and residual.is_contiguous()
    _native.check(L.mdb_conv3d(_native.ptr(x), B, Cin, Z, Y, X, _native.ptr(w), _native.ptr(b), Cout, k, stride,
                               _native.ptr(y), _native.ptr(rb), _native.ptr(residual), _native.ptr(stats),
                               PRECISIONS[precision], _native.current_stream()))
    # statistics are split fixed-point integers inside the library; return them as float64 (sum, sum of squares)
    return (y, words_to_stats(stats)) if want_stats else y


def groupnorm_act(x, stats, gamma, beta, silu=True, precision="bf16"):
    """GroupNorm(32, eps=1e-6) (+SiLU) on NDHWC x using per-channel (sum, sumsq) statistics."""
    L = _native.lib()
    B, C = x.shape[0], x.shape[-1]
    V = x.numel() // (B * C)
    if precision == "bf16x3":
        C //= 2
    y = torch.empty_like(x)
    stats = stats_to_words(stats)
    g = gamma.detach().float().contiguous()
    bt = beta.detach().float().contiguous()
    _native.check(L.mdb_groupnorm_act(_native.ptr(x), _native.ptr(stats), _native.ptr(g), _native.ptr(bt), _native.ptr(y),
                                      B, V, C, 1 if silu else 0, PRECISIONS[precision], _native.current_stream()))
    return y


def sampler_update(eps, x, noise, mask, beta, std, seed=0, offset=0):
    """In-place ancestral update; returns (x, x_mean). eps/x/noise: fp32 [B,C,R,R,R]; mask fp32 [R,R,R]."""
    L = _native.lib()
    B, C = x.shape[0], x.shape[1]
    V = x[0, 0].numel()
    x_mean = torch.empty_like(x)
    _native.check(L.mdb_sampler_update(_native.ptr(eps), _native.ptr(x), _native.ptr(x_mean), _native.ptr(noise),
                                       _native.ptr(mask), float(beta), float(std), V, C, B, seed, offset, None,
                                       _native.current_stream()))
    return x, x_mean


def _train_mode(precision):
    if precision not in ("bf16", "bf16x3"):
        raise ValueError(f"training kernels take precision 'bf16' or 'bf16x3', not {precision!r}")
    return PRECISIONS[precision]


def _parts(precision):
    return 2 if precision == "bf16x3" else 1


def _view_ptr(t, c0):
    """Pointer to channel c0 of an NDHWC bf16 tensor (the hi half of a 'bf16x3' row)."""
    return ctypes.c_void_p(t.data_ptr() + 2 * c0)


def conv3d_backward(dy, x, weight, stride=1, want_dw=True, want_dx=True, precision="bf16", dy_c0=0, x_c0=0, dw=None,
                    accumulate=False, batch=None, splits=1, residual=None):
    """NDHWC conv3d backward: dy [B,Zo,Yo,Xo,*], x [B,Z,Y,X,*] (bf16; 'bf16x3': (hi, lo) rows), weight fp32 OIDHW.

    Returns (dw fp32 OIDHW, dx [B,Z,Y,X,Cin] in the operand layout). Channel views: the operands may be wider than the
    weight's channels (row pitch = their last dimension), read from channel dy_c0 / x_c0 on. `dw` (optional) receives the
    weight gradient, added to it when `accumulate`. The operations are planned for B = x.shape[0] and run for `batch`
    samples (default all). splits > 1 runs the data gradient split-K; `residual` (shaped like dx) is added to dx.
    """
    L = _native.lib()
    mode = _train_mode(precision)
    pp = _parts(precision)
    assert dy.dtype == torch.bfloat16 and x.dtype == torch.bfloat16 and dy.is_contiguous() and x.is_contiguous()
    B, Z, Y, X = x.shape[:4]
    Cout, Cin, k = weight.shape[0], weight.shape[1], weight.shape[2]
    dy_ld, x_ld = dy.shape[-1] // pp, x.shape[-1] // pp
    assert dy_c0 + Cout <= dy_ld and x_c0 + Cin <= x_ld
    w = weight.detach().float().contiguous()
    if dw is None and want_dw:
        dw = torch.zeros_like(w)
    dx = torch.zeros((B, Z, Y, X, Cin * pp), device=x.device, dtype=torch.bfloat16) if want_dx else None
    if residual is not None:
        assert residual.shape == dx.shape and residual.dtype == dx.dtype and residual.is_contiguous()
    _native.check(L.mdb_conv3d_backward(_view_ptr(dy, dy_c0), _view_ptr(x, x_c0), _native.ptr(w), B if batch is None else batch,
                                        Cin, Cout, Z, Y, X, k, stride, _native.ptr(dw), _native.ptr(dx), mode,
                                        0 if dy_ld == Cout else dy_ld, 0 if x_ld == Cin else x_ld, 1 if accumulate else 0, B,
                                        splits, _native.ptr(residual), _native.current_stream()))
    return dw, dx


def groupnorm_act_backward(x, stats, gamma, beta, da, add=None, silu=True, dropout_p=0.0, seed=0, precision="bf16", x1=None,
                           stats1=None, add1=None, dgamma=None, dbeta=None, accumulate=False, want_colsum=False,
                           want_preact=False):
    """Backward of groupnorm_act over the channel concatenation of x and x1 (optional): returns (dx [B,...,C],
    dgamma fp32 [C], dbeta fp32 [C]), then with want_colsum the per-sample column sums of dx fp32 [B, C], and with
    want_preact the pre-activation gradient da * act'(y) * dropout [B,...,C] that the first pass leaves in place of da.

    da, add, add1: dense [B,...,C] in the operand layout. dgamma / dbeta (optional) receive the parameter gradients, added
    to them when `accumulate`.
    """
    L = _native.lib()
    mode = _train_mode(precision)
    pp = _parts(precision)
    B = x.shape[0]
    C0 = x.shape[-1] // pp
    C1 = x1.shape[-1] // pp if x1 is not None else 0
    C = C0 + C1
    V = x.numel() // (B * C0 * pp)
    w0 = stats_to_words(stats)
    w1 = stats_to_words(stats1) if x1 is not None else None
    g = gamma.detach().float().contiguous()
    bt = beta.detach().float().contiguous()
    dx = torch.empty_like(da)
    dg = dgamma if dgamma is not None else torch.empty(C, device=x.device, dtype=torch.float32)
    db = dbeta if dbeta is not None else torch.empty(C, device=x.device, dtype=torch.float32)
    cs = torch.empty((B, C), device=x.device, dtype=torch.float32) if want_colsum else None
    da = da.clone()  # the kernel pair overwrites dL/dy with the pre-activation gradient
    _native.check(L.mdb_groupnorm_act_backward(_native.ptr(x), C0, _native.ptr(x1), C1, _native.ptr(w0), _native.ptr(w1),
                                               _native.ptr(g), _native.ptr(bt), _native.ptr(da), _native.ptr(add),
                                               _native.ptr(add1), _native.ptr(dx), _native.ptr(dg), _native.ptr(db),
                                               _native.ptr(cs), B, V, 1 if silu else 0, float(dropout_p), int(seed), mode,
                                               1 if accumulate else 0, _native.current_stream()))
    return (dx, dg, db) + ((cs,) if want_colsum else ()) + ((da,) if want_preact else ())


def conv3d_dgrad_gn_backward(dy, weight, x, stats, gamma, beta, x1=None, stats1=None, add=None, add1=None, silu=True,
                             dropout_p=0.0, seed=0, precision="bf16"):
    """The training plan's fused path: the data gradient of a k = 3 (stride 1) or k = 1 convolution (weight fp32 OIDHW
    [Cout][C][k^3], dy [B,R,R,R,Cout]) feeds the GroupNorm(+SiLU)(+dropout) backward over x (and x1) in the GEMM epilogue.
    Returns (dx, dgamma, dbeta) like groupnorm_act_backward(x, ..., da=<the data gradient>)."""
    L = _native.lib()
    mode = _train_mode(precision)
    pp = _parts(precision)
    B, R = x.shape[0], x.shape[1]
    C0 = x.shape[-1] // pp
    C1 = x1.shape[-1] // pp if x1 is not None else 0
    C = C0 + C1
    Cout, k = weight.shape[0], weight.shape[2]
    assert weight.shape[1] == C and dy.shape[-1] == Cout * pp and dy.is_contiguous()
    w = weight.detach().float().contiguous()
    w0 = stats_to_words(stats)
    w1 = stats_to_words(stats1) if x1 is not None else None
    g = gamma.detach().float().contiguous()
    bt = beta.detach().float().contiguous()
    dx = torch.empty((B, R, R, R, C * pp), device=x.device, dtype=torch.bfloat16)
    dg = torch.empty(C, device=x.device, dtype=torch.float32)
    db = torch.empty(C, device=x.device, dtype=torch.float32)
    _native.check(L.mdb_conv3d_dgrad_gn_backward(_native.ptr(dy), _native.ptr(w), B, Cout, R, k, _native.ptr(x), C0,
                                                 _native.ptr(x1), C1, _native.ptr(w0), _native.ptr(w1), _native.ptr(g),
                                                 _native.ptr(bt), _native.ptr(add), _native.ptr(add1), _native.ptr(dx),
                                                 _native.ptr(dg), _native.ptr(db), 1 if silu else 0, float(dropout_p),
                                                 int(seed), mode, _native.current_stream()))
    return dx, dg, db


def colsum(t, precision="bf16", c0=0, channels=None, total=None, accumulate=False, from_per=None):
    """Column sums of a [B,...,ld] NDHWC tensor (optionally the channel view [c0, c0 + channels)): returns (per-sample
    sums fp32 [B, C], total fp32 [C]); `total` (optional) is added to when `accumulate`. from_per: per-sample sums
    [B, >= C] fp32 already computed (only the batch sum runs)."""
    L = _native.lib()
    mode = _train_mode(precision)
    pp = _parts(precision)
    B, ld = t.shape[0], t.shape[-1] // pp
    C = ld - c0 if channels is None else channels
    V = t.numel() // (B * ld * pp)
    per = torch.empty((B, C), device=t.device, dtype=torch.float32)
    tot = total if total is not None else torch.empty(C, device=t.device, dtype=torch.float32)
    _native.check(L.mdb_colsum(_view_ptr(t, c0), ld, C, B, V, _native.ptr(per), C, _native.ptr(tot), 1 if accumulate else 0,
                               _native.ptr(from_per), from_per.shape[-1] if from_per is not None else 0, mode,
                               _native.current_stream()))
    return per, tot


def downsum2x(dup, precision="bf16"):
    """Upsample backward: [B,2R,2R,2R,C] -> the sums of its 2x2x2 blocks [B,R,R,R,C]."""
    L = _native.lib()
    B, R2, Cp = dup.shape[0], dup.shape[1], dup.shape[-1]
    dx = torch.empty((B, R2 // 2, R2 // 2, R2 // 2, Cp), device=dup.device, dtype=torch.bfloat16)
    _native.check(L.mdb_downsum2x(_native.ptr(dup), _native.ptr(dx), B, R2 // 2, Cp // _parts(precision), _train_mode(precision),
                                  _native.current_stream()))
    return dx


def batch_sum(t, precision="bf16"):
    """[B,...,C] -> the sum over the batch [...,C]."""
    L = _native.lib()
    B, Cp = t.shape[0], t.shape[-1]
    out = torch.empty(t.shape[1:], device=t.device, dtype=torch.bfloat16)
    _native.check(L.mdb_batch_sum(_native.ptr(t), _native.ptr(out), B, t[0].numel() // Cp, Cp // _parts(precision),
                                  _train_mode(precision), _native.current_stream()))
    return out


def zero_stuff2x(dy, precision="bf16"):
    """[B,R,R,R,C] -> [B,2R,2R,2R,C] holding dy at the odd sites of every axis and zeros elsewhere."""
    L = _native.lib()
    B, R, Cp = dy.shape[0], dy.shape[1], dy.shape[-1]
    z = torch.empty((B, 2 * R, 2 * R, 2 * R, Cp), device=dy.device, dtype=torch.bfloat16)
    _native.check(L.mdb_zero_stuff2x(_native.ptr(dy), _native.ptr(z), B, R, Cp // _parts(precision), _train_mode(precision),
                                     _native.current_stream()))
    return z


def softmax_bwd_rows(P, dP, precision="bf16"):
    """Attention softmax backward in place on dP (fp32 [rows, L]); P: fp32 [rows, L] slots holding the probabilities as
    bf16 at the start of each row ('bf16x3': L hi then L lo). Returns dP, whose rows then hold dS in P's format."""
    L = _native.lib()
    assert P.dtype == torch.float32 and dP.dtype == torch.float32 and P.shape == dP.shape
    _native.check(L.mdb_softmax_bwd_rows(_native.ptr(P), _native.ptr(dP), P.shape[0], P.shape[1], _train_mode(precision),
                                         _native.current_stream()))
    return dP


def transpose_vc(t, c0, channels, precision="bf16"):
    """t [B, V, ld] bf16 operand matrix -> [B, channels, V] of its channels [c0, c0 + channels) ('bf16x3': rows
    [ld hi | ld lo] -> [V hi | V lo])."""
    L = _native.lib()
    pp = _parts(precision)
    B, V, ld = t.shape[0], t.shape[1], t.shape[2] // pp
    out = torch.empty((B, channels, V * pp), device=t.device, dtype=torch.bfloat16)
    _native.check(L.mdb_transpose_vc(_native.ptr(t), ld, c0, _native.ptr(out), B, V, channels, _train_mode(precision),
                                     _native.current_stream()))
    return out


def im2col(x, ksize, kpad, precision="bf16"):
    """fp32 NCDHW [B,Cin,R,R,R] -> [B, R^3, kpad] (column cin*k^3 + tap, zero padded) in the operand layout."""
    L = _native.lib()
    B, Cin, R = x.shape[0], x.shape[1], x.shape[2]
    xc = x.float().contiguous()
    a = torch.empty((B, R ** 3, kpad * _parts(precision)), device=x.device, dtype=torch.bfloat16)
    _native.check(L.mdb_im2col(_native.ptr(xc), _native.ptr(a), B, Cin, R, ksize, kpad, _train_mode(precision),
                               _native.current_stream()))
    return a

"""Operator-level parity of the training kernels in both training operand modes, bf16 and split bf16 ("bf16x3"): the
tcgen05 weight-gradient kernel, the data-gradient GEMMs (single CTA, CTA pair, pointwise, split-K, stride 2), the
two-pass and the fused GroupNorm backward, and the bandwidth kernels of the backward pass.

Every case builds its inputs in fp32, hands them to the kernel through ops.to_ndhwc, and computes the reference in
float64 from the values the kernel actually sees (hi + lo in bf16x3, the bf16 values in bf16). Outputs in split layout
are compared as hi + lo. Errors are max |got - ref| / max |ref|, and every case prints them.

Gates, from the arithmetic (u = 2^-8, the unit roundoff of bf16):
- bf16x3 GEMM outputs (weight and data gradients, the fused GroupNorm backward): a value is carried as hi + lo, off by at
  most u^2 = 2^-16 relative; a product is hi*hi + hi*lo + lo*hi, the dropped lo*lo term is below u^2 of it; the fp32
  accumulation adds 2^-24 per step and a split store u^2 once. Over 10^3-10^4 products of random sign these stay near
  1e-5 of the output scale: gate 1e-4, the same as the forward bf16x3 convolution (tests/test_gpu_conv.py, measured
  6e-6 to 5.6e-5).
- bf16x3 bandwidth kernels (GroupNorm backward, column and batch sums, 2x2x2 block sums, softmax backward): fp32
  arithmetic on exact hi + lo inputs, results stored once as hi + lo (u^2, and 2^-17 on average) or in fp32: gate 2e-5.
- The GroupNorm parameter gradients of the two-pass backward (dgamma, dbeta): sums over B*V elements of the fp32
  pre-activation gradient, taken before it is stored, in a fixed-order staged reduction. Rounding errors of the sum and of
  each element are random and average out to well below 1e-6; a systematic error of the SiLU derivative does not: gate
  1e-6. (The tanh.approx form that suffices for bf16 measured 1.7e-6 to 2.8e-6 here.)
- Every bf16x3 result must also be at least 20 times closer to the float64 result of the data than the bf16 mode of
  the same kernel on the same data (whose operands alone are off by u = 4e-3): this fails if the lo parts are dropped
  anywhere on the way.
- bf16 results against the reference of their own (bf16) operands: fp32 outputs 2e-4, bf16-stored outputs 1e-2.
- Kernels that only move data (zero-stuffing, the operand transposes, im2col) must be bitwise equal to the expected
  tensor.
"""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

X3_GEMM, X3_BW, X3_GN_PARAM, BF16_F32, BF16_STORED, RATIO = 1e-4, 2e-5, 1e-6, 2e-4, 1e-2, 20.0


def _ops():
    from meshdiffusion_b200 import ops
    return ops


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _seen(t, precision):
    """Operand-layout NDHWC tensor -> float64 of the values the kernel reads (hi + lo for 'bf16x3')."""
    if precision == "bf16x3":
        C = t.shape[-1] // 2
        return t[..., :C].double() + t[..., C:].double()
    return t.double()


def _nc(t):
    return t.permute(0, 4, 1, 2, 3).contiguous()


def _nd(t):
    return t.permute(0, 2, 3, 4, 1).contiguous()


def _w_seen(w, precision):
    """The weights as the GEMM packs them: bf16, or a (hi, lo) pair."""
    if precision == "bf16x3":
        hi = w.bfloat16()
        return hi.double() + (w - hi.float()).bfloat16().double()
    return w.bfloat16().double()


def _err(got, ref):
    return (got.double() - ref).abs().max().item() / max(ref.abs().max().item(), 1e-300)


def _check(label, got3, ref3, got16, ref16, gate3, gate16):
    """got3 / ref3: the bf16x3 result and the float64 reference of its operands (= the data to 2^-16); got16 / ref16 the
    same for the bf16 mode. Returns the errors."""
    e3, e16, e16d = _err(got3, ref3), _err(got16, ref16), _err(got16, ref3)
    ratio = e16d / max(e3, 1e-300)
    print(f"{label}: bf16x3 {e3:.3e} (gate {gate3:.0e}); bf16 {e16:.3e} vs its operands, {e16d:.3e} vs the data; "
          f"bf16 / bf16x3 {ratio:.0f}x")
    assert e3 < gate3, f"{label}: bf16x3 error {e3:.3e}"
    assert e16 < gate16, f"{label}: bf16 error {e16:.3e}"
    assert ratio >= RATIO, f"{label}: bf16x3 only {ratio:.1f}x more accurate than bf16"
    return e3


def _conv_grads(x, w, dy, k, stride):
    """float64 autograd of nn.Conv3d (stride 1 'same', or the Downsample pad-high stride 2), NCDHW."""
    x = x.detach().clone().requires_grad_(True)
    w = w.detach().clone().requires_grad_(True)
    y = F.conv3d(x, w, padding=k // 2) if stride == 1 else F.conv3d(F.pad(x, (0, 1, 0, 1, 0, 1)), w, stride=2)
    y.backward(dy)
    return w.grad, x.grad


# ------------------------------------------------------------------------------------------------ weight gradients
WGRAD = [
    # id: (B, Cin, Cout, R, k, stride, options); M = Cout (dY channels), N = Cin (X channels)
    ("flat_k1_192rows_M64_N96", (3, 96, 64, 4, 1, 1, {})),
    ("halo_s1_R16", (2, 128, 128, 16, 3, 1, {})),
    ("groups27_R4_oddB_split2", (3, 128, 128, 4, 3, 1, {})),
    ("stride2_parity_maps", (2, 128, 128, 16, 3, 2, {})),
    ("M512_N512_R4_unsplit", (1, 512, 512, 4, 3, 1, {})),
    ("M96_N192_R8", (2, 192, 96, 8, 3, 1, {})),
    ("R32_geometry", (1, 64, 64, 32, 3, 1, {})),
    ("channel_views", (2, 128, 128, 8, 3, 1, {"x_ld": 256, "x_c0": 64, "dy_ld": 192, "dy_c0": 32})),
    ("accumulate", (2, 128, 64, 8, 3, 1, {"accumulate": True})),
    ("batch3_of_planned4", (4, 128, 128, 4, 3, 1, {"batch": 3})),
    ("flat_batch2_of_planned3", (3, 64, 128, 8, 1, 1, {"batch": 2})),
]


@pytest.mark.parametrize("case", [c for _, c in WGRAD], ids=[i for i, _ in WGRAD])
def test_wgrad(case):
    ops = _ops()
    B, Cin, Cout, R, k, stride, o = case
    Ro = R // stride
    x_ld, x_c0 = o.get("x_ld", Cin), o.get("x_c0", 0)
    dy_ld, dy_c0 = o.get("dy_ld", Cout), o.get("dy_c0", 0)
    nb, acc = o.get("batch", B), o.get("accumulate", False)
    g = _gen(B * 7919 + Cin * 31 + Cout + R)
    x = torch.randn(B, x_ld, R, R, R, device="cuda", generator=g)
    dy = torch.randn(B, dy_ld, Ro, Ro, Ro, device="cuda", generator=g)
    w = torch.randn(Cout, Cin, k, k, k, device="cuda", generator=g) / (Cin * k ** 3) ** 0.5
    prefill = torch.randn(w.shape, device="cuda", generator=g) if acc else None
    out = {}
    for prec in ("bf16x3", "bf16"):
        xi, dyi = ops.to_ndhwc(x, prec), ops.to_ndhwc(dy, prec)
        dw, _ = ops.conv3d_backward(dyi, xi, w, stride=stride, want_dx=False, precision=prec, dy_c0=dy_c0, x_c0=x_c0,
                                    dw=prefill.clone() if acc else None, accumulate=acc, batch=nb)
        xs = _nc(_seen(xi, prec)[:nb, ..., x_c0:x_c0 + Cin])
        dys = _nc(_seen(dyi, prec)[:nb, ..., dy_c0:dy_c0 + Cout])
        ref = _conv_grads(xs, w.double(), dys, k, stride)[0]
        if acc:
            ref = ref + prefill.double()
        out[prec] = (dw, ref)
    _check(f"wgrad {case[:6]} {o}", *out["bf16x3"], *out["bf16"], X3_GEMM, BF16_F32)


# ------------------------------------------------------------------------------------------------ data gradients
DGRAD = [
    # id: (B, Cin, Cout, R, k, stride, options); dx has the Cin channels of the forward convolution
    ("single_cta_R16", (2, 64, 128, 16, 3, 1, {})),
    ("cta_pair_R32_B3", (3, 128, 128, 32, 3, 1, {})),
    ("pointwise", (2, 128, 256, 8, 1, 1, {})),
    ("split_k4", (2, 256, 512, 4, 3, 1, {"splits": 4})),
    ("split_k4_residual", (2, 256, 512, 4, 3, 1, {"splits": 4, "residual": True})),
    ("stride2_zero_stuffed", (2, 128, 128, 16, 3, 2, {})),
]


@pytest.mark.parametrize("case", [c for _, c in DGRAD], ids=[i for i, _ in DGRAD])
def test_dgrad(case):
    ops = _ops()
    B, Cin, Cout, R, k, stride, o = case
    Ro = R // stride
    g = _gen(B * 131 + Cin + Cout * 7 + R)
    x = torch.randn(B, Cin, R, R, R, device="cuda", generator=g)  # only its shape is used
    dy = torch.randn(B, Cout, Ro, Ro, Ro, device="cuda", generator=g)
    w = torch.randn(Cout, Cin, k, k, k, device="cuda", generator=g) / (Cout * k ** 3) ** 0.5
    res = torch.randn(B, Cin, R, R, R, device="cuda", generator=g) if o.get("residual") else None
    out = {}
    for prec in ("bf16x3", "bf16"):
        dyi = ops.to_ndhwc(dy, prec)
        ri = ops.to_ndhwc(res, prec) if res is not None else None
        _, dx = ops.conv3d_backward(dyi, ops.to_ndhwc(x, prec), w, stride=stride, want_dw=False, precision=prec,
                                    splits=o.get("splits", 1), residual=ri)
        ref = _conv_grads(x.double(), _w_seen(w, prec), _nc(_seen(dyi, prec)), k, stride)[1]
        if ri is not None:
            ref = ref + _nc(_seen(ri, prec))
        out[prec] = (_nc(_seen(dx, prec)), ref)
    _check(f"dgrad {case[:6]} {o}", *out["bf16x3"], *out["bf16"], X3_GEMM, BF16_STORED)


# ------------------------------------------------------------------------------------------------ GroupNorm backward
def _drop_keep(B, V, C, p, seed):
    """The kernels' dropout mask, [B, V, C] bool: element e = (b*V + v)*C + c is kept iff
    ((hash(seed, e >> 2) >> 16*(e & 3)) & 0xFFFF) >= round(p * 65536), hash = backward.cuh::drop_hash64 (splitmix64)."""
    def u64(v):
        return v - (1 << 64) if v >= (1 << 63) else v

    def shr(z, n):  # logical right shift of an int64 holding a uint64
        return (z >> n) & ((1 << (64 - n)) - 1)

    e = torch.arange(B * V * C, device="cuda", dtype=torch.int64)
    z = (e >> 2) + u64((seed * 0x9E3779B97F4A7C15) % (1 << 64))
    z = (z ^ shr(z, 30)) * u64(0xBF58476D1CE4E5B9)
    z = (z ^ shr(z, 27)) * u64(0x94D049BB133111EB)
    z = z ^ shr(z, 31)
    r16 = (z >> (16 * (e & 3))) & 0xFFFF  # (the sign-extended bits of an arithmetic shift are masked off)
    return (r16 >= round(p * 65536)).view(B, V, C)


def _gn_ref(xs, gamma, beta, da, silu, p, seed, adds):
    """float64 autograd of GroupNorm(32, eps 1e-6) [-> SiLU] [-> dropout] (NCDHW); returns (dx + adds, dgamma, dbeta)."""
    B, C = xs.shape[:2]
    V = xs[0, 0].numel()
    x = xs.detach().clone().requires_grad_(True)
    gm = gamma.double().clone().requires_grad_(True)
    bt = beta.double().clone().requires_grad_(True)
    y = F.group_norm(x, 32, gm, bt, eps=1e-6)
    if silu:
        y = F.silu(y)
    if p > 0:
        keep = _drop_keep(B, V, C, p, seed).permute(0, 2, 1).reshape(xs.shape)
        y = y * keep.double() / (1.0 - p)
    y.backward(da)
    dx = x.grad
    for a in adds:
        dx = dx + a
    return dx, gm.grad, bt.grad


def _stats(xs):
    """float64 [B, C, 2] (sum, sum of squares) of an NDHWC float64 tensor."""
    B, C = xs.shape[0], xs.shape[-1]
    t = xs.reshape(B, -1, C)
    return torch.stack([t.sum(1), (t * t).sum(1)], dim=-1)


GN = [
    # id: (B, R, C0, C1, silu, n_add, dropout, accumulate, colsum)
    ("single_silu_add0", (2, 8, 128, 0, True, 1, 0.0, False, False)),
    ("concat_silu_add01_dropout", (2, 8, 128, 256, True, 2, 0.3, False, False)),
    ("single_nosilu_accumulate_colsum", (3, 8, 256, 0, False, 0, 0.0, True, True)),
    ("concat_nosilu_add0_dropout_colsum", (2, 8, 128, 256, False, 1, 0.3, False, True)),
]


def _gn_inputs(B, R, C0, C1, n_add, seed):
    g = _gen(seed)
    C = C0 + C1
    x = torch.randn(B, C, R, R, R, device="cuda", generator=g) * 1.5 + 0.3
    gamma = torch.rand(C, device="cuda", generator=g) + 0.5
    beta = torch.randn(C, device="cuda", generator=g) * 0.1
    da = torch.randn(B, C, R, R, R, device="cuda", generator=g)
    adds = [torch.randn(B, C, R, R, R, device="cuda", generator=g) for _ in range(n_add)]
    return x, gamma, beta, da, adds


@pytest.mark.parametrize("case", [c for _, c in GN], ids=[i for i, _ in GN])
def test_groupnorm_backward_two_pass(case):
    ops = _ops()
    B, R, C0, C1, silu, n_add, p, acc, want_cs = case
    seed = 0x5EED + C1
    x, gamma, beta, da, adds = _gn_inputs(B, R, C0, C1, n_add, 17 + C0 + C1 + B)
    pre_g = torch.randn(C0 + C1, device="cuda") if acc else None
    pre_b = torch.randn(C0 + C1, device="cuda") if acc else None
    got, ref = {}, {}
    for prec in ("bf16x3", "bf16"):
        x0 = ops.to_ndhwc(x[:, :C0], prec)
        x1 = ops.to_ndhwc(x[:, C0:], prec) if C1 else None
        s0, s1 = _stats(_seen(x0, prec)), (_stats(_seen(x1, prec)) if C1 else None)
        dai = ops.to_ndhwc(da, prec)
        ai = [ops.to_ndhwc(a, prec) for a in adds]
        r = ops.groupnorm_act_backward(x0, s0, gamma, beta, dai, add=ai[0] if n_add > 0 else None, silu=silu, dropout_p=p,
                                       seed=seed, precision=prec, x1=x1, stats1=s1, add1=ai[1] if n_add > 1 else None,
                                       dgamma=pre_g.clone() if acc else None, dbeta=pre_b.clone() if acc else None,
                                       accumulate=acc, want_colsum=want_cs)
        xs = torch.cat([_seen(x0, prec)] + ([_seen(x1, prec)] if C1 else []), dim=-1)
        dx_r, dg_r, db_r = _gn_ref(_nc(xs), gamma, beta, _nc(_seen(dai, prec)), silu, p, seed, [_nc(_seen(a, prec)) for a in ai])
        if acc:
            dg_r, db_r = dg_r + pre_g.double(), db_r + pre_b.double()
        got[prec] = {"dx": _nc(_seen(r[0], prec)), "dgamma": r[1], "dbeta": r[2]}
        ref[prec] = {"dx": dx_r, "dgamma": dg_r, "dbeta": db_r}
        if want_cs:
            got[prec]["colsum"] = r[3]
            ref[prec]["colsum"] = dx_r.sum(dim=(2, 3, 4))
    for k in got["bf16x3"]:
        _check(f"gn two-pass {case} {k}", got["bf16x3"][k], ref["bf16x3"][k], got["bf16"][k], ref["bf16"][k],
               X3_GN_PARAM if k in ("dgamma", "dbeta") else X3_BW, BF16_STORED if k == "dx" else BF16_F32 * 10)


@pytest.mark.parametrize("p", [0.0, 0.3])
def test_groupnorm_backward_silu_derivative_per_element(p):
    """Pass 1 replaces dL/da by dL/dy = da * silu'(y) * dropout element by element. Its error in units of |da| / (1 - p)
    is the error of silu'(y) at that element (|silu'| <= 1.1), over 2^20 elements with |y| up to about 17. bf16x3: the
    (hi, lo) store costs up to 2^-16 * 1.1 = 1.7e-5, the fp32 evaluation of y and silu' a few 2^-22: gate 2e-5. bf16: the
    bf16 store alone is up to 2^-8 * 1.1."""
    ops = _ops()
    B, R, C = 2, 16, 128
    g = _gen(53)
    x = torch.randn(B, C, R, R, R, device="cuda", generator=g) * 1.5 + 0.3
    gamma = torch.rand(C, device="cuda", generator=g) * 3.0 + 0.5
    beta = torch.randn(C, device="cuda", generator=g)
    da = torch.randn(B, C, R, R, R, device="cuda", generator=g)
    keep = _drop_keep(B, R ** 3, C, p, 99).view(B, R, R, R, C) if p > 0 else torch.ones(B, R, R, R, C, dtype=torch.bool, device="cuda")
    errs = {}
    for prec in ("bf16x3", "bf16"):
        xi, dai = ops.to_ndhwc(x, prec), ops.to_ndhwc(da, prec)
        xs = _seen(xi, prec)
        dy = _seen(ops.groupnorm_act_backward(xi, _stats(xs), gamma, beta, dai, silu=True, dropout_p=p, seed=99,
                                              precision=prec, want_preact=True)[-1], prec)
        y = _nd(F.group_norm(_nc(xs), 32, gamma.double(), beta.double(), eps=1e-6))
        s = torch.sigmoid(y)
        scale = _seen(dai, prec).abs() / (1.0 - p)
        ref = _seen(dai, prec) * s * (1.0 + y * (1.0 - s)) / (1.0 - p)
        assert torch.all(dy[~keep] == 0)
        errs[prec] = ((dy - ref).abs() / scale.clamp_min(1e-30))[keep].max().item()
        print(f"silu' per element, p={p}, |y| <= {y.abs().max().item():.1f}: {prec} {errs[prec]:.3e}")
    assert errs["bf16x3"] < 2e-5
    assert errs["bf16"] < 1e-2


FUSED = [
    # id: (B, R, Cout, C0, C1, k, silu, dropout, n_add)
    ("k3_single_silu_R16", (2, 16, 128, 128, 0, 3, True, 0.0, 0)),
    ("k3_concat_silu_dropout_add01", (2, 8, 128, 128, 256, 3, True, 0.3, 2)),
    ("k1_single_nosilu_add0", (2, 8, 256, 128, 0, 1, False, 0.0, 1)),
    ("k3_cta_pair_R32_silu_dropout", (3, 32, 128, 128, 0, 3, True, 0.3, 0)),
]


@pytest.mark.parametrize("case", [c for _, c in FUSED], ids=[i for i, _ in FUSED])
def test_groupnorm_backward_fused(case):
    """The data-gradient GEMM with the GroupNorm-backward epilogue, its tile reduce and the apply pass, against float64;
    and element by element against the unfused pair (the same data gradient stored, then the two-pass backward)."""
    ops = _ops()
    B, R, Cout, C0, C1, k, silu, p, n_add = case
    C = C0 + C1
    seed = 0xD0 + R
    x, gamma, beta, _, adds = _gn_inputs(B, R, C0, C1, n_add, 23 + C + R)
    g = _gen(29 + C + R)
    dy = torch.randn(B, Cout, R, R, R, device="cuda", generator=g)
    w = torch.randn(Cout, C, k, k, k, device="cuda", generator=g) / (Cout * k ** 3) ** 0.5
    got, ref, two = {}, {}, {}
    for prec in ("bf16x3", "bf16"):
        x0 = ops.to_ndhwc(x[:, :C0], prec)
        x1 = ops.to_ndhwc(x[:, C0:], prec) if C1 else None
        s0, s1 = _stats(_seen(x0, prec)), (_stats(_seen(x1, prec)) if C1 else None)
        dyi = ops.to_ndhwc(dy, prec)
        ai = [ops.to_ndhwc(a, prec) for a in adds]
        kw = dict(x1=x1, stats1=s1, add=ai[0] if n_add > 0 else None, add1=ai[1] if n_add > 1 else None, silu=silu,
                  dropout_p=p, seed=seed, precision=prec)
        dx, dg, db = ops.conv3d_dgrad_gn_backward(dyi, w, x0, s0, gamma, beta, **kw)
        _, da = ops.conv3d_backward(dyi, torch.empty(B, R, R, R, C * (2 if prec == "bf16x3" else 1), device="cuda",
                                                     dtype=torch.bfloat16), w, want_dw=False, precision=prec)
        kw.pop("add")
        dx2, dg2, db2 = ops.groupnorm_act_backward(x0, s0, gamma, beta, da, add=ai[0] if n_add > 0 else None, **kw)
        xs = torch.cat([_seen(x0, prec)] + ([_seen(x1, prec)] if C1 else []), dim=-1)
        da_r = _conv_grads(torch.zeros(B, C, R, R, R, device="cuda", dtype=torch.float64), _w_seen(w, prec),
                           _nc(_seen(dyi, prec)), k, 1)[1]
        dx_r, dg_r, db_r = _gn_ref(_nc(xs), gamma, beta, da_r, silu, p, seed, [_nc(_seen(a, prec)) for a in ai])
        got[prec] = {"dx": _nc(_seen(dx, prec)), "dgamma": dg, "dbeta": db}
        ref[prec] = {"dx": dx_r, "dgamma": dg_r, "dbeta": db_r}
        two[prec] = {"dx": _nc(_seen(dx2, prec)), "dgamma": dg2, "dbeta": db2}
    for key in got["bf16x3"]:
        _check(f"gn fused {case} {key}", got["bf16x3"][key], ref["bf16x3"][key], got["bf16"][key], ref["bf16"][key],
               X3_GEMM, BF16_STORED)
    # fused vs two-pass: the only difference is the stored data gradient (split: 2^-16 relative, bf16: 2^-8)
    for prec, gate in (("bf16x3", 5e-5), ("bf16", 2e-2)):
        for key in got[prec]:
            e = _err(got[prec][key], two[prec][key].double())
            print(f"gn fused vs two-pass {case} {prec} {key}: {e:.3e}")
            assert e < gate


# ------------------------------------------------------------------------------------------------ bandwidth kernels
@pytest.mark.parametrize("B,R,ld,c0,C,acc", [(2, 8, 192, 64, 64, False), (3, 16, 128, 0, 128, True)])
def test_colsum(B, R, ld, c0, C, acc):
    ops = _ops()
    g = _gen(B + R + ld)
    t = torch.randn(B, ld, R, R, R, device="cuda", generator=g) + 0.25
    pre = torch.randn(C, device="cuda", generator=g) * 100.0 if acc else None
    got, ref = {}, {}
    for prec in ("bf16x3", "bf16"):
        ti = ops.to_ndhwc(t, prec)
        per, tot = ops.colsum(ti, prec, c0=c0, channels=C, total=pre.clone() if acc else None, accumulate=acc)
        per_r = _seen(ti, prec)[..., c0:c0 + C].sum(dim=(1, 2, 3))
        tot_r = per_r.sum(0) + (pre.double() if acc else 0)
        got[prec], ref[prec] = (per, tot), (per_r, tot_r)
        # the producer-supplied path: only the batch sum runs, on the given per-sample sums (pitch 2C)
        fp = torch.randn(B, 2 * C, device="cuda", generator=g)
        per2, tot2 = ops.colsum(ti, prec, c0=c0, channels=C, from_per=fp)
        e = _err(tot2, fp[:, :C].double().sum(0))
        assert torch.equal(per2, fp[:, :C]) and e < 1e-6, e
    _check(f"colsum per B{B} R{R} ld{ld} c0{c0}", got["bf16x3"][0], ref["bf16x3"][0], got["bf16"][0], ref["bf16"][0], X3_BW, BF16_F32)
    _check(f"colsum total acc={acc}", got["bf16x3"][1], ref["bf16x3"][1], got["bf16"][1], ref["bf16"][1], X3_BW, BF16_F32)


def test_downsum2x():
    ops = _ops()
    B, R, C = 2, 8, 64
    t = torch.randn(B, C, 2 * R, 2 * R, 2 * R, device="cuda", generator=_gen(41))
    got, ref = {}, {}
    for prec in ("bf16x3", "bf16"):
        ti = ops.to_ndhwc(t, prec)
        got[prec] = _nc(_seen(ops.downsum2x(ti, prec), prec))
        ref[prec] = _nc(_seen(ti, prec)).view(B, C, R, 2, R, 2, R, 2).sum(dim=(3, 5, 7))
    _check("downsum2x", got["bf16x3"], ref["bf16x3"], got["bf16"], ref["bf16"], X3_BW, BF16_STORED)


def test_batch_sum():
    ops = _ops()
    B, R, C = 3, 8, 128
    t = torch.randn(B, C, R, R, R, device="cuda", generator=_gen(43))
    got, ref = {}, {}
    for prec in ("bf16x3", "bf16"):
        ti = ops.to_ndhwc(t, prec)
        got[prec] = _seen(ops.batch_sum(ti, prec)[None], prec)
        ref[prec] = _seen(ti, prec).sum(0, keepdim=True)
    _check("batch_sum", got["bf16x3"], ref["bf16x3"], got["bf16"], ref["bf16"], X3_BW, BF16_STORED)


@pytest.mark.parametrize("rows,L", [(128, 512), (6, 4096)])
def test_softmax_backward(rows, L):
    ops = _ops()
    g = _gen(rows + L)
    prob = torch.softmax(torch.randn(rows, L, device="cuda", generator=g) * 3.0, dim=-1)
    dP = torch.randn(rows, L, device="cuda", generator=g)
    got, ref = {}, {}
    for prec in ("bf16x3", "bf16"):
        P = torch.zeros(rows, L, device="cuda")
        hi = prob.bfloat16()
        P.view(torch.bfloat16)[:, :L] = hi
        ps = hi.double()
        if prec == "bf16x3":
            lo = (prob - hi.float()).bfloat16()
            P.view(torch.bfloat16)[:, L:] = lo
            ps = ps + lo.double()
        d = ops.softmax_bwd_rows(P, dP.clone(), prec).view(torch.bfloat16)
        ds = d[:, :L].double() + (d[:, L:].double() if prec == "bf16x3" else 0)
        got[prec] = ds
        ref[prec] = ps * (dP.double() - (ps * dP.double()).sum(-1, keepdim=True))
    _check(f"softmax backward rows {rows} L {L}", got["bf16x3"], ref["bf16x3"], got["bf16"], ref["bf16"], X3_BW, BF16_STORED)


@pytest.mark.parametrize("precision", ["bf16", "bf16x3"])
def test_zero_stuff2x_bitwise(precision):
    ops = _ops()
    B, R, C = 2, 8, 64
    dy = ops.to_ndhwc(torch.randn(B, C, R, R, R, device="cuda", generator=_gen(47)), precision)
    z = ops.zero_stuff2x(dy, precision)
    want = torch.zeros_like(z)
    want[:, 1::2, 1::2, 1::2] = dy
    assert torch.equal(z.view(torch.int16), want.view(torch.int16))


@pytest.mark.parametrize("precision", ["bf16", "bf16x3"])
@pytest.mark.parametrize("V,ld,c0,C", [(512, 384, 128, 128), (512, 384, 0, 128), (512, 192, 64, 96), (4096, 128, 0, 128)])
def test_transpose_bitwise(precision, V, ld, c0, C):
    """The attention backward's operand transposes (fast 64x64 path, and the generic one for C = 96)."""
    ops = _ops()
    B = 2
    pp = 2 if precision == "bf16x3" else 1
    t = torch.randn(B, V, ld * pp, device="cuda", generator=_gen(V + ld + c0)).bfloat16()
    out = ops.transpose_vc(t, c0, C, precision)
    want = t[:, :, c0:c0 + C].transpose(1, 2)
    if precision == "bf16x3":
        want = torch.cat([want, t[:, :, ld + c0:ld + c0 + C].transpose(1, 2)], dim=-1)
    assert torch.equal(out.view(torch.int16), want.contiguous().view(torch.int16))


@pytest.mark.parametrize("precision", ["bf16", "bf16x3"])
@pytest.mark.parametrize("Cin,R,k", [(4, 16, 3), (4, 32, 5), (1, 16, 3)])
def test_im2col_bitwise(precision, Cin, R, k):
    """The stem / head im2col: column cin*k^3 + tap, tap = (kd*k + kh)*k + kw, zero padding k/2, padded to a multiple of 64."""
    ops = _ops()
    B, p, T = 2, k // 2, k ** 3
    Kpad = (Cin * T + 63) // 64 * 64
    x = torch.randn(B, Cin, R, R, R, device="cuda", generator=_gen(Cin + R + k))
    a = ops.im2col(x, k, Kpad, precision)
    xp = F.pad(x, (p,) * 6)
    cols = torch.stack([xp[:, :, kd:kd + R, kh:kh + R, kw:kw + R] for kd in range(k) for kh in range(k) for kw in range(k)], dim=2)
    cols = cols.permute(0, 3, 4, 5, 1, 2).reshape(B, R ** 3, Cin * T)
    cols = F.pad(cols, (0, Kpad - Cin * T))
    hi = cols.bfloat16()
    want = torch.cat([hi, (cols - hi.float()).bfloat16()], dim=-1) if precision == "bf16x3" else hi
    assert torch.equal(a.view(torch.int16), want.view(torch.int16))


def test_training_kernels_refuse_tf32():
    from meshdiffusion_b200 import _native
    ops = _ops()
    x = torch.zeros(1, 4, 4, 4, 32, device="cuda", dtype=torch.bfloat16)
    with pytest.raises(ValueError):
        ops.zero_stuff2x(x, "tf32")
    L = _native.lib()
    rc = L.mdb_zero_stuff2x(_native.ptr(x), _native.ptr(torch.empty(1, 8, 8, 8, 32, device="cuda", dtype=torch.bfloat16)),
                            1, 4, 32, 1, _native.current_stream())
    assert rc != 0 and b"precision" in L.mdb_last_error()

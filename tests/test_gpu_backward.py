"""Training path parity on the GPU: the tcgen05 weight-gradient kernel, the data-gradient convolutions, GroupNorm
backward and the whole score-network backward, against torch autograd in true fp32 (the reference computes its
gradients with `loss.backward()`, lib/diffusion/losses.py:104-139).

bf16 operands: the kernels see bf16-rounded inputs, which the fp32 autograd reference is given too, so weight
gradients (fp32 accumulation) agree to ~1e-4; bf16-stored activation gradients to bf16 resolution.
"""
import pytest
import torch
import torch.nn.functional as F

from helpers import build_model, rel_l2, rel_max, tiny_config
from oracle import synth, unet_oracle

pytestmark = pytest.mark.gpu


def _ndhwc(t):
    return t.permute(0, 2, 3, 4, 1).contiguous().to(torch.bfloat16)


CONV_CASES = [
    # (B, Cin, Cout, R, k, stride)
    (2, 64, 128, 16, 3, 1),    # (8,16,1,1) tiles, halo reuse, one Cout tile
    (1, 256, 128, 16, 3, 1),   # two Cin tiles
    (3, 128, 256, 8, 3, 1),    # (8,8,2,1) tiles, per-tap loads
    (3, 128, 128, 4, 3, 1),    # (4,4,4,2) tiles, odd batch -> half-empty tile
    (2, 32, 32, 16, 3, 1),     # channel chunks padded by TMA zero fill
    (2, 128, 128, 16, 3, 2),   # Downsample: stride 2, parity sub-grids
    (3, 96, 64, 4, 1, 1),      # pointwise, 192 rows (partial last tile)
    (2, 128, 512, 8, 1, 1),    # pointwise, 4 Cout tiles
]


@pytest.mark.parametrize("B,Cin,Cout,R,k,stride", CONV_CASES)
def test_conv3d_backward(B, Cin, Cout, R, k, stride):
    from meshdiffusion_b200 import ops
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    g = torch.Generator(device="cuda").manual_seed(B * 1000 + Cin + R)
    x = torch.randn(B, Cin, R, R, R, device="cuda", generator=g).bfloat16().float().requires_grad_(True)
    w = (torch.randn(Cout, Cin, k, k, k, device="cuda", generator=g) / (Cin * k ** 3) ** 0.5).requires_grad_(True)
    wq = w.detach().bfloat16().float()
    if stride == 1:
        y = F.conv3d(x, w, None, padding=k // 2)
    else:
        y = F.conv3d(F.pad(x, (0, 1, 0, 1, 0, 1)), w, None, stride=2)
    dy = torch.randn(y.shape, device="cuda", generator=g).bfloat16().float()
    y.backward(dy)
    want_dx = stride == 1
    dw, dx = ops.conv3d_backward(_ndhwc(dy), _ndhwc(x.detach()), w.detach(), stride=stride, want_dx=want_dx)
    e_w = rel_max(dw, w.grad)
    print(f"wgrad B{B} {Cin}->{Cout} R{R} k{k} s{stride}: max {e_w:.3e}")
    assert e_w < 2e-4
    if want_dx:
        # the kernel multiplies by bf16-rounded weights: reference data gradient with the same rounding
        xr = x.detach().clone().requires_grad_(True)
        F.conv3d(xr, wq, None, padding=k // 2).backward(dy)
        got = dx.float().permute(0, 4, 1, 2, 3)
        e_x = rel_max(got, xr.grad)
        print(f"dgrad: max {e_x:.3e}")
        assert e_x < 6e-3


@pytest.mark.parametrize("C,R,B,silu,with_add", [(128, 16, 2, True, False), (32, 8, 3, True, True), (384, 8, 2, False, True), (1024, 4, 2, True, False)])
def test_groupnorm_act_backward(C, R, B, silu, with_add):
    from meshdiffusion_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(C + R)
    x = (torch.randn(B, C, R, R, R, device="cuda", generator=g) * 1.5 + 0.3).bfloat16().float().requires_grad_(True)
    gamma = (torch.rand(C, device="cuda", generator=g) + 0.5).requires_grad_(True)
    beta = (torch.randn(C, device="cuda", generator=g) * 0.1).requires_grad_(True)
    y = F.group_norm(x, 32, gamma, beta, eps=1e-6)
    if silu:
        y = F.silu(y)
    da = torch.randn(y.shape, device="cuda", generator=g).bfloat16().float()
    y.backward(da)
    add = torch.randn(x.shape, device="cuda", generator=g).bfloat16().float() if with_add else None
    xl = _ndhwc(x.detach())
    xd = xl.double().reshape(B, -1, C)
    stats = torch.stack([xd.sum(1), (xd * xd).sum(1)], dim=-1)
    dx, dg, db = ops.groupnorm_act_backward(xl, stats, gamma.detach(), beta.detach(), _ndhwc(da), _ndhwc(add) if with_add else None, silu=silu)
    ref_dx = x.grad + (add if with_add else 0)
    e = rel_max(dx.float().permute(0, 4, 1, 2, 3), ref_dx)
    eg, eb = rel_max(dg, gamma.grad), rel_max(db, beta.grad)
    print(f"gn bwd C{C} R{R}: dx {e:.3e} dgamma {eg:.3e} dbeta {eb:.3e}")
    assert e < 1e-2 and eg < 2e-3 and eb < 2e-3


def _oracle_grads(cfg, sd, x, labels, noise, mask, amp=False):
    """fp32 autograd through the oracle network with the reference's DDPM loss (losses.py:69-78). `amp`: the same graph
    under torch's bf16 autocast (what stock PyTorch does for a bf16 training run of these modules)."""
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    sdg = {k: (v.cuda().clone().requires_grad_(True) if v.dtype == torch.float32 and k not in ("mask", "coords") else v.cuda()) for k, v in sd.items()}
    arch = unet_oracle.arch_from_config(cfg)
    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=amp):
        pred = unet_oracle.unet_forward(sdg, arch, x, labels)
    pred = pred.float()
    losses = torch.square(pred - noise) * mask
    losses = losses.reshape(losses.shape[0], -1).mean(dim=-1)
    loss = torch.mean(losses) / mask.sum() * mask.numel()
    loss.backward()
    return loss.detach(), pred.detach(), {k: v.grad for k, v in sdg.items() if v.dtype == torch.float32 and v.requires_grad and v.grad is not None}


@pytest.mark.parametrize("name", ["res64", "res128"])
def test_unet_backward_matches_autograd(name):
    cfg = tiny_config(name, "bf16")
    cfg.model.dropout = 0.0
    model, sd = build_model(cfg, "cuda:0", 21)
    net = model.module
    R, B = cfg.data.image_size, 2
    x, labels = synth.synthetic_inputs(R, B, 31, sd["mask"])
    x, labels = x.cuda(), labels.cuda()
    gen = torch.Generator(device="cuda").manual_seed(5)
    noise = torch.randn(x.shape, device="cuda", generator=gen)
    mask = sd["mask"].cuda().view(1, 1, R, R, R)
    ref_loss, ref_pred, ref = _oracle_grads(cfg, sd, x, labels, noise, mask)

    net.train()
    pred = model(x, labels)
    losses = (torch.square(pred - noise) * mask).reshape(B, -1).mean(dim=-1)
    loss = torch.mean(losses) / mask.sum() * mask.numel()
    loss.backward()
    print(f"{name}: loss {loss.item():.6f} vs {ref_loss.item():.6f}; pred rel-l2 {rel_l2(pred.detach(), ref_pred):.3e}")
    assert abs(loss.item() - ref_loss.item()) < 3e-2 * abs(ref_loss.item())
    rows, tot_num, tot_den = [], 0.0, 0.0
    for n, p in net.named_parameters():
        if n in ("mask", "coords") or n not in ref:
            continue
        assert p.grad is not None, n
        gr = ref[n]
        num = (p.grad - gr).double().pow(2).sum().item()
        den = gr.double().pow(2).sum().item()
        tot_num += num; tot_den += den
        rows.append((n, num, den, p.grad.double().pow(2).sum().item()))
    glob = (tot_num / tot_den) ** 0.5
    # Tensors whose true gradient vanishes (pos_layer.weight sees coords*0; the attention KEY bias NIN_1.b shifts every
    # logit of a row equally, which softmax ignores) carry only rounding noise in the fp32 reference: they are checked
    # for being negligible, the others for their relative error.
    checked, worst = 0, ("", 0.0)
    for n, num, den, ours in rows:
        if den < 1e-10 * tot_den:
            assert ours < 1e-6 * tot_den, f"{n}: gradient should vanish, got norm^2 {ours:.3e} of {tot_den:.3e}"
            continue
        e = (num / den) ** 0.5
        checked += 1
        if e > worst[1]:
            worst = (n, e)
    print(f"{name}: {checked}/{len(rows)} tensors, global rel-l2 {glob:.3e}, worst {worst[0]} {worst[1]:.3e}")
    assert glob < 3e-2 and worst[1] < 1e-1


def _global_rel_l2(grads, ref):
    num = sum((grads[n] - g).double().pow(2).sum().item() for n, g in ref.items() if n in grads)
    den = sum(g.double().pow(2).sum().item() for n, g in ref.items() if n in grads)
    return (num / den) ** 0.5


@pytest.mark.parametrize("name", ["res64", "res128"])
def test_backward_error_not_above_stock_bf16_autocast(name):
    """BASELINE config 3 trains in bf16. The yardstick for a bf16 backward is what stock PyTorch makes of the SAME modules
    under bf16 autocast: both are compared with true-fp32 autograd, and the native gradients must not be further from it
    than the autocast ones (measured: native ~1.2e-2, autocast ~1.6e-2 global rel-l2 on the test networks)."""
    cfg = tiny_config(name, "bf16")
    cfg.model.dropout = 0.0
    model, sd = build_model(cfg, "cuda:0", 23)
    net = model.module
    R, B = cfg.data.image_size, 2
    x, labels = synth.synthetic_inputs(R, B, 37, sd["mask"])
    x, labels = x.cuda(), labels.cuda()
    noise = torch.randn(x.shape, device="cuda", generator=torch.Generator(device="cuda").manual_seed(9))
    mask = sd["mask"].cuda().view(1, 1, R, R, R)
    _, _, ref = _oracle_grads(cfg, sd, x, labels, noise, mask)
    _, _, amp = _oracle_grads(cfg, sd, x, labels, noise, mask, amp=True)
    net.train()
    pred = model(x, labels)
    losses = (torch.square(pred - noise) * mask).reshape(B, -1).mean(dim=-1)
    (torch.mean(losses) / mask.sum() * mask.numel()).backward()
    ours = {n: p.grad for n, p in net.named_parameters() if p.grad is not None}
    e_native, e_amp = _global_rel_l2(ours, ref), _global_rel_l2(amp, ref)
    print(f"{name}: gradient global rel-l2 vs fp32 autograd: native bf16 {e_native:.3e}, torch bf16 autocast {e_amp:.3e}")
    assert e_native < 1.25 * e_amp + 2e-3


def test_unet_backward_accumulates_and_is_deterministic():
    cfg = tiny_config("res64", "bf16")
    cfg.model.dropout = 0.0
    model, sd = build_model(cfg, "cuda:0", 3)
    net = model.module
    net.train()
    R, B = 16, 2
    x, labels = synth.synthetic_inputs(R, B, 8, sd["mask"])
    x, labels = x.cuda(), labels.cuda()

    def run():
        out = model(x, labels)
        out.square().mean().backward()

    run()
    g1 = net._flat_grad.clone()
    for p in net.parameters():
        p.grad = None
    run()
    assert torch.equal(g1, net._flat_grad), "gradients differ run to run"
    run()  # second micro-batch without zero_grad: accumulation (losses.py:111-113)
    assert torch.allclose(net._flat_grad, 2 * g1, rtol=1e-5, atol=1e-8)


def test_train_step_fn_reduces_loss():
    """The reference's step_fn / optimize_fn / EMA loop runs unchanged on the engine: a few steps on one batch."""
    from meshdiffusion_b200.diffusion import losses, sde_lib
    from meshdiffusion_b200.diffusion.models import ema as ema_lib
    cfg = tiny_config("res64", "bf16")
    cfg.model.dropout = 0.1
    cfg.optim.lr = 2e-4
    cfg.optim.warmup = 0
    torch.manual_seed(0)
    model, sd = build_model(cfg, "cuda:0", 9)
    net = model.module
    R, B = 16, 4
    mask = sd["mask"].cuda().view(1, 1, R, R, R)
    sde = sde_lib.VPSDE(cfg.model.beta_min, cfg.model.beta_max, cfg.model.num_scales, device="cuda:0")
    optimizer = losses.get_optimizer(cfg, model.parameters())
    ema = ema_lib.ExponentialMovingAverage(model.parameters(), decay=cfg.model.ema_rate)
    state = dict(optimizer=optimizer, model=model, ema=ema, step=0)
    step_fn = losses.get_step_fn(sde, train=True, optimize_fn=losses.optimization_manager(cfg), mask=mask)
    g = torch.Generator(device="cuda").manual_seed(2)
    batch = torch.randn(B, 4, R, R, R, device="cuda", generator=g).clamp(-1, 1) * mask
    first = []
    for it in range(12):
        first.append(step_fn(state, batch)["loss"].item())
    print("losses:", " ".join(f"{v:.4f}" for v in first))
    assert all(torch.isfinite(torch.tensor(first)))
    assert sum(first[-4:]) / 4 < sum(first[:4]) / 4, "loss did not go down"
    assert state["step"] == 12


def test_loss_curve_tracks_fp32_reference():
    """SURVEY 8(d)-3: 20 optimiser steps with dropout disabled, same data / labels / noise / Adam settings, engine (bf16
    operands) vs fp32 autograd through the oracle network: the loss curves must stay together."""
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    cfg = tiny_config("res64", "bf16")
    cfg.model.dropout = 0.0
    model, sd = build_model(cfg, "cuda:0", 13)
    net = model.module
    net.train()
    R, B, steps = 16, 4, 20
    mask = sd["mask"].cuda().view(1, 1, R, R, R)
    arch = unet_oracle.arch_from_config(cfg)
    ref_sd = {k: (v.cuda().clone().requires_grad_(True) if v.dtype == torch.float32 and k not in ("mask", "coords") else v.cuda()) for k, v in sd.items()}
    ref_params = [v for v in ref_sd.values() if v.requires_grad]
    opt_ref = torch.optim.Adam(ref_params, lr=2e-4, betas=(0.9, 0.999), eps=1e-8)
    opt = torch.optim.Adam([p for p in net.parameters() if p.requires_grad], lr=2e-4, betas=(0.9, 0.999), eps=1e-8)
    g = torch.Generator(device="cuda").manual_seed(4)
    data = (torch.rand(B, 4, R, R, R, device="cuda", generator=g) * 2 - 1) * mask

    def ddpm_loss(pred, noise):
        l = (torch.square(pred - noise) * mask).reshape(B, -1).mean(dim=-1)
        return torch.mean(l) / mask.sum() * mask.numel()

    ours, theirs = [], []
    for it in range(steps):
        labels = torch.randint(0, 1000, (B,), device="cuda", generator=g).float()
        noise = torch.randn(data.shape, device="cuda", generator=g)
        x = (0.7 * data + 0.7 * noise) * mask
        opt_ref.zero_grad()
        lr_ = ddpm_loss(unet_oracle.unet_forward(ref_sd, arch, x, labels), noise)
        lr_.backward()
        torch.nn.utils.clip_grad_norm_(ref_params, 1.0)
        opt_ref.step()
        opt.zero_grad()
        lo = ddpm_loss(model(x, labels), noise)
        lo.backward()
        torch.nn.utils.clip_grad_norm_([p for p in net.parameters() if p.requires_grad], 1.0)
        opt.step()
        ours.append(lo.item()); theirs.append(lr_.item())
    print("engine:", " ".join(f"{v:.4f}" for v in ours))
    print("fp32  :", " ".join(f"{v:.4f}" for v in theirs))
    rel = max(abs(a - b) / abs(b) for a, b in zip(ours, theirs))
    print(f"max relative loss difference over {steps} steps: {rel:.3e}")
    assert rel < 5e-2
    assert theirs[-1] < theirs[0]


@pytest.mark.parametrize("name", ["res64", "res128"])
def test_unet_backward_matches_reference_golden(name):
    """Engine gradients vs the signatures (norm + 4 random projections per tensor) of the REFERENCE modules' own
    loss.backward() on CPU fp32 (oracle/make_golden.py::golden_unet_backward)."""
    import numpy as np
    from helpers import ddpm_loss, grad_signature, load_golden
    gold = load_golden(f"unet_tiny_{name}_grads.npz")
    cfg = tiny_config(name, "bf16")
    cfg.model.dropout = 0.0
    model, sd = build_model(cfg, "cuda:0", int(gold["state_seed"]))
    net = model.module
    net.train()
    R = cfg.data.image_size
    x, labels = synth.synthetic_inputs(R, 2, int(gold["input_seed"]), sd["mask"])
    noise = torch.randn(x.shape, generator=torch.Generator().manual_seed(int(gold["noise_seed"]))).cuda()
    loss = ddpm_loss(model(x.cuda(), labels.cuda()), noise, sd["mask"].cuda().view(1, 1, R, R, R))
    loss.backward()
    print(f"{name}: loss {loss.item():.6f} vs reference {float(gold['loss']):.6f}")
    assert abs(loss.item() - float(gold["loss"])) < 2e-2 * float(gold["loss"])
    tot = float(gold["total_norm"])
    params = dict(net.named_parameters())
    worst = 0.0
    for n, sig in zip(gold["names"], gold["sig"]):
        got = grad_signature(str(n), params[str(n)].grad)
        # a projection of the error onto a unit-variance random vector is ~ N(0, |err|^2): 4 sigma of a 5 % error
        tol = 4 * (0.05 * sig[0] + 2e-3 * tot)
        assert abs(got[0] - sig[0]) < 0.1 * sig[0] + 2e-3 * tot, f"{n}: norm {got[0]:.4e} vs {sig[0]:.4e}"
        assert np.abs(got[1:] - sig[1:]).max() < tol, f"{n}: projections {got[1:]} vs {sig[1:]}"
        worst = max(worst, np.abs(got[1:] - sig[1:]).max() / tot)
    print(f"{name}: {len(gold['names'])} tensors, worst projection error / |g| {worst:.3e}")


def test_res64_full_backward_vs_autograd():
    """Full-size network (64^3 ... 4^3 levels, CTA-pair data gradients, 16-way split weight gradients, both attention
    resolutions): every gradient tensor against fp32 autograd through the oracle, B = 1."""
    from helpers import ddpm_loss, full_config
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    cfg = full_config("res64", "bf16")
    cfg.model.dropout = 0.0
    model, sd = build_model(cfg, "cuda:0", 5)
    net = model.module
    net.train()
    R = 64
    x, labels = synth.synthetic_inputs(R, 1, 6, sd["mask"])
    x, labels = x.cuda(), labels.cuda()
    noise = torch.randn(x.shape, device="cuda", generator=torch.Generator(device="cuda").manual_seed(9))
    mask = sd["mask"].cuda().view(1, 1, R, R, R)
    loss = ddpm_loss(model(x, labels), noise, mask)
    loss.backward()
    ours = {n: p.grad.clone() for n, p in net.named_parameters() if p.grad is not None}
    net.release_engine()
    torch.cuda.empty_cache()
    osd = {k: (v.cuda().clone().requires_grad_(True) if v.dtype == torch.float32 and k not in ("mask", "coords") else v.cuda()) for k, v in sd.items()}
    ref_loss = ddpm_loss(unet_oracle.unet_forward(osd, unet_oracle.arch_from_config(cfg), x, labels), noise, mask)
    ref_loss.backward()
    assert abs(loss.item() - ref_loss.item()) < 3e-2 * abs(ref_loss.item())
    tot_num = tot_den = 0.0
    rows = []
    for n, g in ours.items():
        if n not in osd or osd[n].grad is None:
            continue
        num = (g - osd[n].grad).double().pow(2).sum().item()
        den = osd[n].grad.double().pow(2).sum().item()
        tot_num += num; tot_den += den
        rows.append((n, num, den))
    glob = (tot_num / tot_den) ** 0.5
    worst = max(((n, (num / den) ** 0.5) for n, num, den in rows if den > 1e-8 * tot_den), key=lambda t: t[1])
    print(f"res64 full: loss {loss.item():.5f} vs {ref_loss.item():.5f}; {len(rows)} tensors, global rel-l2 {glob:.3e}, worst {worst[0]} {worst[1]:.3e}")
    assert glob < 4e-2 and worst[1] < 1.5e-1


def test_dropout_gradients_fused_vs_two_pass(monkeypatch):
    """Dropout masks come from a counter hash of (seed, layer, element) evaluated in three places: the forward
    GroupNorm-apply kernel, the two-pass GroupNorm backward, and the fused GEMM epilogue. With a fixed seed the fused and
    the two-pass engines must therefore produce the same gradients (up to bf16 rounding of dy), which pins the element
    indexing of all three against each other; and the gradients must differ from the no-dropout ones."""
    import ctypes
    from meshdiffusion_b200 import _native
    cfg = tiny_config("res64", "bf16")
    cfg.model.dropout = 0.3
    R, B = 16, 2

    def grads(fused, p):
        monkeypatch.setenv("MDB_GNB", "1" if fused else "0")
        torch.manual_seed(1234)  # the dropout seed derives from torch.initial_seed() and a per-model call counter
        cfg.model.dropout = p
        model, sd = build_model(cfg, "cuda:0", 3)
        net = model.module
        net.train()
        x, labels = synth.synthetic_inputs(R, B, 8, sd["mask"])
        model(x.cuda(), labels.cuda()).square().mean().backward()
        g = net._flat_grad.clone()
        net.release_engine()
        return g

    g_fused, g_two = grads(True, 0.3), grads(False, 0.3)
    g_none = grads(True, 0.0)
    rel = (g_fused - g_two).norm().item() / g_two.norm().item()
    away = (g_fused - g_none).norm().item() / g_none.norm().item()
    print(f"fused vs two-pass under dropout: rel-l2 {rel:.3e}; dropout vs none: {away:.3e}")
    assert rel < 1e-2
    assert away > 5e-2


def test_backward_with_smaller_runtime_batch():
    """An engine planned for batch 4 must give, for a batch of 2, the gradients of an engine planned for 2 (weight-gradient
    tensor maps / split plans and the tile-partial rows are re-derived per runtime batch). Not bitwise: the split-K plan of
    the small GEMMs depends on the planned batch, which changes fp32 summation order before the bf16 stores."""
    cfg = tiny_config("res64", "bf16")
    cfg.model.dropout = 0.0
    R = 16

    def run(first_batch):
        model, sd = build_model(cfg, "cuda:0", 3)
        net = model.module
        net.train()
        x, labels = synth.synthetic_inputs(R, 4, 8, sd["mask"])
        x, labels = x.cuda(), labels.cuda()
        if first_batch == 4:
            model(x, labels).square().mean().backward()
            for p in net.parameters():
                p.grad = None
        model(x[:2].contiguous(), labels[:2].contiguous()).square().mean().backward()
        g = net._flat_grad.clone()
        net.release_engine()
        return g

    g4, g2 = run(4), run(2)
    rel = (g4 - g2).norm().item() / g2.norm().item()
    print(f"planned-4 vs planned-2 engines on a batch of 2: rel-l2 {rel:.3e}")
    assert rel < 1e-2


def test_res64_full_loss_curve_tracks_fp32_reference():
    """The 20-step tiny-network experiment at the real size: 8 Adam steps of the full res64 network (batch 2, dropout off)
    on the engine vs fp32 autograd through the oracle with identical data, labels and noise."""
    from helpers import ddpm_loss, full_config
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    cfg = full_config("res64", "bf16")
    cfg.model.dropout = 0.0
    model, sd = build_model(cfg, "cuda:0", 5)
    net = model.module
    net.train()
    R, B, steps = 64, 2, 8
    mask = sd["mask"].cuda().view(1, 1, R, R, R)
    arch = unet_oracle.arch_from_config(cfg)
    ref_sd = {k: (v.cuda().clone().requires_grad_(True) if v.dtype == torch.float32 and k not in ("mask", "coords") else v.cuda()) for k, v in sd.items()}
    ref_params = [v for v in ref_sd.values() if v.requires_grad]
    opt_ref = torch.optim.Adam(ref_params, lr=1e-4)
    opt = torch.optim.Adam([p for p in net.parameters() if p.requires_grad], lr=1e-4)
    g = torch.Generator(device="cuda").manual_seed(4)
    data = (torch.rand(B, 4, R, R, R, device="cuda", generator=g) * 2 - 1) * mask
    ours, theirs = [], []
    for it in range(steps):
        labels = torch.randint(0, 1000, (B,), device="cuda", generator=g).float()
        noise = torch.randn(data.shape, device="cuda", generator=g)
        x = (0.7 * data + 0.7 * noise) * mask
        opt_ref.zero_grad()
        lr_ = ddpm_loss(unet_oracle.unet_forward(ref_sd, arch, x, labels), noise, mask)
        lr_.backward()
        torch.nn.utils.clip_grad_norm_(ref_params, 1.0)
        opt_ref.step()
        opt.zero_grad()
        lo = ddpm_loss(model(x, labels), noise, mask)
        lo.backward()
        torch.nn.utils.clip_grad_norm_([p for p in net.parameters() if p.requires_grad], 1.0)
        opt.step()
        ours.append(lo.item()); theirs.append(lr_.item())
    print("engine:", " ".join(f"{v:.4f}" for v in ours))
    print("fp32  :", " ".join(f"{v:.4f}" for v in theirs))
    rel = max(abs(a - b) / abs(b) for a, b in zip(ours, theirs))
    print(f"max relative loss difference over {steps} full-size steps: {rel:.3e}")
    # lr 1e-4 without warm-up halves the loss within four steps; bf16 operands track the fp32 trajectory to ~2 % through
    # that transient (6e-4 in the gentler tiny-network experiment) and, above all, stay finite: the pre-GroupNorm
    # activations grow to an rms of several hundred here, which is what exposed the statistics overflow
    assert all(torch.isfinite(torch.tensor(ours)))
    assert rel < 4e-2
    assert abs(ours[-1] - theirs[-1]) < 2e-2 * theirs[-1]

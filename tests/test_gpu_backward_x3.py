"""Split-bf16 ("bf16x3") training plan on the GPU: forward, data gradients (with the fused GroupNorm-backward epilogue),
weight gradients and the bandwidth kernels of the backward pass in (hi, lo) operands, against fp32 autograd through the
oracle network and against the reference's own CPU fp32 `loss.backward()` signatures. The gates follow from the
arithmetic (products carry ~2^-16 relative error instead of bf16's 2^-8); every measured figure is printed.
"""
import os

import pytest
import torch

from helpers import ROOT, build_model, ddpm_loss, tiny_config
from oracle import synth, unet_oracle

pytestmark = pytest.mark.gpu

# Gradient error against fp32 autograd, as relative L2 over all tensors and for the worst single tensor. Measured on one
# B200 (1000 W power limit): global 3.9e-5 / 3.7e-5 / 4.9e-5, worst tensor 6.3e-5 / 9.4e-5 / 1.1e-4 (tiny res64, tiny
# res128, full res64). The gates leave margin above that and stay well below the error one split kernel brings when it
# drops its lo parts: zeroing them in the batch sum of the stem (global 2.0e-4, worst 1.8e-3) or the bias column sums
# (worst 2.4e-3) passed the former gates of 1e-3 / 1e-2.
GLOBAL_GATE, WORST_GATE = 2e-4, 1e-3


def _cfg(name="res64", precision="bf16x3"):
    cfg = tiny_config(name, "bf16")
    cfg.training.compute_dtype = precision
    cfg.model.dropout = 0.0
    return cfg


def _errors(grads, ref):
    """(global rel-L2, (worst tensor, its rel-L2)) over the tensors whose reference gradient does not vanish."""
    rows, num_t, den_t = [], 0.0, 0.0
    for n, g in grads.items():
        if n not in ref:
            continue
        num = (g - ref[n]).double().pow(2).sum().item()
        den = ref[n].double().pow(2).sum().item()
        num_t += num; den_t += den
        rows.append((n, num, den))
    worst = max(((n, (num / den) ** 0.5) for n, num, den in rows if den > 1e-10 * den_t), key=lambda t: t[1])
    return (num_t / den_t) ** 0.5, worst


def _oracle_grads(cfg, sd, x, labels, noise, mask):
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    sdg = {k: (v.cuda().clone().requires_grad_(True) if v.dtype == torch.float32 and k not in ("mask", "coords") else v.cuda()) for k, v in sd.items()}
    loss = ddpm_loss(unet_oracle.unet_forward(sdg, unet_oracle.arch_from_config(cfg), x, labels), noise, mask)
    loss.backward()
    return loss.item(), {k: v.grad for k, v in sdg.items() if v.dtype == torch.float32 and v.requires_grad and v.grad is not None}


def _engine_grads(cfg, state_seed, x, labels, noise, mask):
    model, _ = build_model(cfg, "cuda:0", state_seed)
    net = model.module
    net.train()
    loss = ddpm_loss(model(x, labels), noise, mask)
    loss.backward()
    grads = {n: p.grad.clone() for n, p in net.named_parameters() if p.grad is not None}
    net.release_engine()
    return loss.item(), grads


@pytest.mark.parametrize("name", ["res64", "res128"])
def test_x3_gradients_match_fp32_autograd(name):
    cfg = _cfg(name)
    _, sd = build_model(cfg, "cuda:0", 21)
    R, B = cfg.data.image_size, 2
    x, labels = synth.synthetic_inputs(R, B, 31, sd["mask"])
    x, labels = x.cuda(), labels.cuda()
    noise = torch.randn(x.shape, device="cuda", generator=torch.Generator(device="cuda").manual_seed(5))
    mask = sd["mask"].cuda().view(1, 1, R, R, R)
    ref_loss, ref = _oracle_grads(cfg, sd, x, labels, noise, mask)
    loss, ours = _engine_grads(cfg, 21, x, labels, noise, mask)
    _, ours_bf16 = _engine_grads(_cfg(name, "bf16"), 21, x, labels, noise, mask)
    glob, worst = _errors(ours, ref)
    glob16, worst16 = _errors(ours_bf16, ref)
    print(f"{name}: loss {loss:.6f} vs {ref_loss:.6f}; bf16x3 global rel-l2 {glob:.3e}, worst {worst[0]} {worst[1]:.3e}; "
          f"bf16 engine global {glob16:.3e}, worst {worst16[1]:.3e}; ratio {glob16 / glob:.1f}x")
    assert abs(loss - ref_loss) < 1e-3 * abs(ref_loss)
    assert glob < GLOBAL_GATE and worst[1] < WORST_GATE
    assert glob * 10 <= glob16


@pytest.mark.parametrize("name", ["res64", "res128"])
def test_x3_gradients_match_reference_golden(name):
    """Against the signatures (norm + 4 random projections per tensor) of the reference modules' own CPU fp32
    loss.backward() (tests/golden/unet_tiny_*_grads.npz), with tolerances 5x (norms) / 10x (projections) tighter than
    the bf16 plan's."""
    import numpy as np
    from helpers import grad_signature, load_golden
    gold = load_golden(f"unet_tiny_{name}_grads.npz")
    cfg = _cfg(name)
    model, sd = build_model(cfg, "cuda:0", int(gold["state_seed"]))
    net = model.module
    net.train()
    R = cfg.data.image_size
    x, labels = synth.synthetic_inputs(R, 2, int(gold["input_seed"]), sd["mask"])
    noise = torch.randn(x.shape, generator=torch.Generator().manual_seed(int(gold["noise_seed"]))).cuda()
    loss = ddpm_loss(model(x.cuda(), labels.cuda()), noise, sd["mask"].cuda().view(1, 1, R, R, R))
    loss.backward()
    print(f"{name}: loss {loss.item():.7f} vs reference {float(gold['loss']):.7f}")
    assert abs(loss.item() - float(gold["loss"])) < 1e-3 * float(gold["loss"])
    tot = float(gold["total_norm"])
    params = dict(net.named_parameters())
    worst_n = worst_p = 0.0
    for n, sig in zip(gold["names"], gold["sig"]):
        got = grad_signature(str(n), params[str(n)].grad)
        assert abs(got[0] - sig[0]) < 1e-2 * sig[0] + 2e-4 * tot, f"{n}: norm {got[0]:.6e} vs {sig[0]:.6e}"
        assert np.abs(got[1:] - sig[1:]).max() < 4 * (5e-3 * sig[0] + 2e-4 * tot), f"{n}: projections {got[1:]} vs {sig[1:]}"
        worst_n = max(worst_n, abs(got[0] - sig[0]) / tot)
        worst_p = max(worst_p, np.abs(got[1:] - sig[1:]).max() / tot)
    print(f"{name}: {len(gold['names'])} tensors, worst norm error / |g| {worst_n:.3e}, worst projection error / |g| {worst_p:.3e}")


def test_x3_res64_full_backward_vs_autograd():
    """Full-size res64 (CTA-pair X3 data gradients with the GroupNorm-backward epilogue, split weight gradients, both
    attention resolutions), B = 1: every gradient tensor against fp32 autograd through the oracle."""
    from helpers import full_config
    cfg = full_config("res64", "bf16")
    cfg.training.compute_dtype = "bf16x3"
    cfg.model.dropout = 0.0
    _, sd = build_model(cfg, "cuda:0", 5)
    R = 64
    x, labels = synth.synthetic_inputs(R, 1, 6, sd["mask"])
    x, labels = x.cuda(), labels.cuda()
    noise = torch.randn(x.shape, device="cuda", generator=torch.Generator(device="cuda").manual_seed(9))
    mask = sd["mask"].cuda().view(1, 1, R, R, R)
    loss, ours = _engine_grads(cfg, 5, x, labels, noise, mask)
    torch.cuda.empty_cache()
    ref_loss, ref = _oracle_grads(cfg, sd, x, labels, noise, mask)
    glob, worst = _errors(ours, ref)
    print(f"res64 full bf16x3: loss {loss:.6f} vs {ref_loss:.6f}; global rel-l2 {glob:.3e}, worst {worst[0]} {worst[1]:.3e}")
    assert abs(loss - ref_loss) < 1e-3 * abs(ref_loss)
    assert glob < GLOBAL_GATE and worst[1] < WORST_GATE


def test_x3_loss_curve_tracks_fp32_reference():
    """20 Adam steps (dropout off, same data / labels / noise / Adam settings): engine in bf16x3 vs fp32 autograd."""
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    cfg = _cfg()
    model, sd = build_model(cfg, "cuda:0", 13)
    net = model.module
    net.train()
    R, B, steps = 16, 4, 20
    mask = sd["mask"].cuda().view(1, 1, R, R, R)
    arch = unet_oracle.arch_from_config(cfg)
    ref_sd = {k: (v.cuda().clone().requires_grad_(True) if v.dtype == torch.float32 and k not in ("mask", "coords") else v.cuda()) for k, v in sd.items()}
    ref_params = [v for v in ref_sd.values() if v.requires_grad]
    opt_ref = torch.optim.Adam(ref_params, lr=2e-4, betas=(0.9, 0.999), eps=1e-8)
    params = [p for p in net.parameters() if p.requires_grad]
    opt = torch.optim.Adam(params, lr=2e-4, betas=(0.9, 0.999), eps=1e-8)
    g = torch.Generator(device="cuda").manual_seed(4)
    data = (torch.rand(B, 4, R, R, R, device="cuda", generator=g) * 2 - 1) * mask
    ours, theirs = [], []
    for _ in range(steps):
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
        torch.nn.utils.clip_grad_norm_(params, 1.0)
        opt.step()
        ours.append(lo.item()); theirs.append(lr_.item())
    print("engine:", " ".join(f"{v:.5f}" for v in ours))
    print("fp32  :", " ".join(f"{v:.5f}" for v in theirs))
    rel = max(abs(a - b) / abs(b) for a, b in zip(ours, theirs))
    print(f"bf16x3: max relative loss difference over {steps} steps: {rel:.3e}")
    assert rel < 5e-3
    assert theirs[-1] < theirs[0]


def test_x3_backward_accumulates_and_is_deterministic():
    cfg = _cfg()
    model, sd = build_model(cfg, "cuda:0", 3)
    net = model.module
    net.train()
    x, labels = synth.synthetic_inputs(16, 2, 8, sd["mask"])
    x, labels = x.cuda(), labels.cuda()

    def run():
        model(x, labels).square().mean().backward()

    run()
    g1 = net._flat_grad.clone()
    for p in net.parameters():
        p.grad = None
    run()
    assert torch.equal(g1, net._flat_grad), "gradients differ run to run"
    run()  # second micro-batch without zero_grad: accumulation
    assert torch.allclose(net._flat_grad, 2 * g1, rtol=1e-5, atol=1e-8)


def test_x3_backward_with_smaller_runtime_batch():
    """An engine planned for batch 4 must give, for a batch of 2, the gradients of an engine planned for 2."""
    cfg = _cfg()

    def run(first_batch):
        model, sd = build_model(cfg, "cuda:0", 3)
        net = model.module
        net.train()
        x, labels = synth.synthetic_inputs(16, 4, 8, sd["mask"])
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
    print(f"bf16x3 planned-4 vs planned-2 engines on a batch of 2: rel-l2 {rel:.3e}")
    assert rel < 1e-4


def test_x3_dropout_gradients_fused_vs_two_pass(monkeypatch):
    """The split-bf16 GroupNorm-apply kernel draws the same dropout hash, at the same element index, as the two backward
    paths (fused GEMM epilogue, two-pass GroupNorm backward): with a fixed seed both engines agree, and the gradients
    differ from the no-dropout ones."""
    cfg = _cfg()

    def grads(fused, p):
        monkeypatch.setenv("MDB_GNB", "1" if fused else "0")
        torch.manual_seed(1234)  # the dropout seed derives from torch.initial_seed() and a per-model call counter
        cfg.model.dropout = p
        model, sd = build_model(cfg, "cuda:0", 3)
        net = model.module
        net.train()
        x, labels = synth.synthetic_inputs(16, 2, 8, sd["mask"])
        model(x.cuda(), labels.cuda()).square().mean().backward()
        g = net._flat_grad.clone()
        net.release_engine()
        return g

    g_fused, g_two = grads(True, 0.3), grads(False, 0.3)
    g_none = grads(True, 0.0)
    rel = (g_fused - g_two).norm().item() / g_two.norm().item()
    away = (g_fused - g_none).norm().item() / g_none.norm().item()
    print(f"bf16x3 fused vs two-pass under dropout: rel-l2 {rel:.3e}; dropout vs none: {away:.3e}")
    assert rel < 1e-4
    assert away > 5e-2


def test_x3_train_step_fn_reduces_loss():
    """The product step (losses.get_step_fn, FusedAdam, EMA) with the split-bf16 plan: 12 steps on one batch."""
    from meshdiffusion_b200.diffusion import losses, sde_lib
    from meshdiffusion_b200.diffusion.models import ema as ema_lib
    cfg = _cfg()
    cfg.model.dropout = 0.1
    cfg.optim.lr = 2e-4
    cfg.optim.warmup = 0
    torch.manual_seed(0)
    model, sd = build_model(cfg, "cuda:0", 9)
    assert model.module.train_precision == "bf16x3"
    R, B = 16, 4
    mask = sd["mask"].cuda().view(1, 1, R, R, R)
    sde = sde_lib.VPSDE(cfg.model.beta_min, cfg.model.beta_max, cfg.model.num_scales, device="cuda:0")
    optimizer = losses.get_optimizer(cfg, model.parameters())
    ema = ema_lib.ExponentialMovingAverage(model.parameters(), decay=cfg.model.ema_rate)
    state = dict(optimizer=optimizer, model=model, ema=ema, step=0)
    step_fn = losses.get_step_fn(sde, train=True, optimize_fn=losses.optimization_manager(cfg), mask=mask)
    batch = torch.randn(B, 4, R, R, R, device="cuda", generator=torch.Generator(device="cuda").manual_seed(2)).clamp(-1, 1) * mask
    first = [step_fn(state, batch)["loss"].item() for _ in range(12)]
    print("bf16x3 losses:", " ".join(f"{v:.4f}" for v in first))
    assert all(torch.isfinite(torch.tensor(first)))
    assert sum(first[-4:]) / 4 < sum(first[:4]) / 4, "loss did not go down"
    assert state["step"] == 12


def test_x3_train_cli_writes_reference_checkpoint_layout(tmp_path):
    """`main_diffusion.py --mode=train --config.training.compute_dtype=bf16x3`: three optimiser steps, then the
    checkpoint files of the reference's trainer."""
    import subprocess
    import sys
    import numpy as np
    wd = os.path.join(tmp_path, "run")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "main_diffusion.py"), f"--config={ROOT}/configs/res64.py", "--mode=train",
                        f"--config.training.train_dir={wd}", "--config.data.synthetic=True", "--config.training.batch_size=1",
                        "--config.training.n_iters=3", "--config.training.log_freq=1", "--config.training.snapshot_freq_for_preemption=2",
                        "--config.training.snapshot_freq=100000", "--config.training.compute_dtype=bf16x3"],
                       cwd=str(tmp_path), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    ck = torch.load(os.path.join(wd, "checkpoints-meta", "checkpoint.pth"), map_location="cpu", weights_only=False)
    assert set(ck.keys()) == {"optimizer", "model", "ema", "step"}
    losses = [float(l.split("training_loss:")[1]) for l in (r.stderr + r.stdout).splitlines() if "training_loss:" in l]
    print("bf16x3 CLI losses:", losses)
    assert len(losses) >= 3 and all(np.isfinite(losses))
    final = torch.load(os.path.join(wd, "checkpoints", "checkpoint_3.pth"), map_location="cpu", weights_only=False)
    assert final["step"] == 4


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_x3_two_rank_overlapped_allreduce_matches_single_rank_double_batch(tmp_path):
    import subprocess
    import sys
    import test_gpu_multi
    child = test_gpu_multi.CHILD.replace('cfg.model.dropout = 0.0\n', 'cfg.model.dropout = 0.0\ncfg.training.compute_dtype = "bf16x3"\n')
    child = child.replace("assert err < 1e-3, err", "assert err < 1e-4, err")
    assert child.count("bf16x3") == 1 and "err < 1e-4" in child
    script = os.path.join(tmp_path, "dp_child_x3.py")
    open(script, "w").write(child)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29543", script],
                       capture_output=True, text=True, timeout=600)
    print(r.stdout[-2000:])
    assert r.returncode == 0, r.stderr[-3000:]
    assert r.stdout.count("DP_RANK_OK") == 2 and "DP_GRAD_REL_L2" in r.stdout

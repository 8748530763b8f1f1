"""CPU: host-side pieces of the drop-in surface compared with what the REFERENCE's own code computes (stored in
tests/golden/reference_host.json.xz by oracle/make_host_golden.py): config trees key by key, registered predictor / corrector /
model names, the VP-SDE tables and `marginal_prob`, the EMA recursion, the optimiser construction and the warm-up / clip
arithmetic of `optimization_manager` (lib/diffusion/losses.py:26-52)."""
import json
import lzma
import os

import numpy as np
import pytest
import torch

from helpers import GOLD


@pytest.fixture(scope="module")
def ref():
    return json.load(lzma.open(os.path.join(GOLD, "reference_host.json.xz"), "rt"))


def _flat(c, pre=""):
    o = {}
    for k, v in c.items():
        if k == "device":
            continue
        if isinstance(v, dict):
            o.update(_flat(v, pre + k + "."))
        else:
            o[pre + k] = list(v) if isinstance(v, tuple) else v
    return o


@pytest.mark.parametrize("name", ["res64", "res128"])
def test_config_tree_has_every_reference_key_with_its_value(ref, name):
    from configs import res64, res128
    ours = _flat((res128 if name == "res128" else res64).get_config())
    theirs = ref[name]
    missing = sorted(set(theirs) - set(ours))
    assert not missing, f"reference config keys absent here: {missing}"
    diff = {k: (ours[k], v) for k, v in theirs.items() if ours[k] != v}
    assert not diff, f"values differ from the reference's configs/{name}.py: {diff}"
    # keys only this repository has must be additions of its own (engine knobs), never renamed reference keys
    extra = sorted(set(ours) - set(theirs))
    assert all(k.split(".")[-1] in ("compute_dtype", "engine_max_batch", "grad_overlap", "grad_bucket_mb", "synthetic", "native_rng",
                                    "normalize_sdf", "extension", "deform_scale") or k == "seed" for k in extra), extra


def test_registries_hold_the_reference_names(ref):
    from meshdiffusion_b200.diffusion import sampling
    from meshdiffusion_b200.diffusion.models import ddpm, utils as mutils  # noqa: F401  (registers the models)
    for n in ref["predictors"]:
        assert sampling.get_predictor(n) is not None, n
    for n in ref["correctors"]:
        assert sampling.get_corrector(n) is not None, n
    for n in ref["models"]:
        assert mutils.get_model(n) is not None, n


def test_vpsde_tables_and_marginal_prob_equal_the_reference(ref):
    from configs import res64
    from meshdiffusion_b200.diffusion import sde_lib
    cfg = res64.get_config()
    sde = sde_lib.VPSDE(beta_min=cfg.model.beta_min, beta_max=cfg.model.beta_max, N=cfg.model.num_scales, device="cpu")
    for n in ("discrete_betas", "alphas", "alphas_cumprod", "sqrt_alphas_cumprod", "sqrt_1m_alphas_cumprod"):
        assert np.array_equal(getattr(sde, n).double().numpy(), np.array(ref["sde"][n])), n  # bit-equal fp32 tables
    x = torch.linspace(-1, 1, 24).view(2, 3, 4)
    mean, std = sde.marginal_prob(x, torch.tensor([0.25, 0.9]))
    assert np.array_equal(mean.double().numpy(), np.array(ref["sde"]["mp_mean"]))
    assert np.array_equal(std.double().numpy(), np.array(ref["sde"]["mp_std"]))


def test_ema_recursion_equals_the_reference(ref):
    from meshdiffusion_b200.diffusion.models.ema import ExponentialMovingAverage
    p = [torch.nn.Parameter(torch.arange(6, dtype=torch.float32))]
    ema = ExponentialMovingAverage(p, decay=0.9999)
    for want in ref["ema"]:
        p[0].data.mul_(1.5).add_(0.25)
        ema.update(p)
        assert np.array_equal(ema.shadow_params[0].double().numpy(), np.array(want))


def test_optimizer_defaults_equal_the_reference(ref):
    """`get_optimizer` builds an Adam with the reference's hyper-parameters (the fused step itself needs the GPU and is pinned
    against torch.optim.Adam in tests/test_gpu_train_ops.py); the warm-up schedule is the reference's lr * min(step / warmup, 1)."""
    from configs import res64
    from meshdiffusion_b200.diffusion import losses
    cfg = res64.get_config()
    w = [torch.nn.Parameter(torch.zeros(5, 3)), torch.nn.Parameter(torch.zeros(7))]
    opt = losses.get_optimizer(cfg, w)
    assert isinstance(opt, torch.optim.Adam)
    for k, v in ref["optim"]["defaults"].items():
        ours = opt.defaults[k]
        assert (list(ours) if isinstance(ours, tuple) else ours) == v, k
    for step, rec in zip((0, 10, 4999, 20000), ref["optim"]["steps"]):
        want = cfg.optim.lr * min(step / cfg.optim.warmup, 1.0) if cfg.optim.warmup > 0 else cfg.optim.lr
        assert abs(rec["lr"] - want) <= 1e-12 * max(abs(want), 1e-30), (step, rec["lr"], want)


def test_sigmas_buffer_equals_the_reference(ref):
    from configs import res64
    from meshdiffusion_b200.diffusion.models import utils as mutils
    ours = mutils.get_sigmas(res64.get_config())
    assert np.array_equal(np.asarray(ours, dtype=np.float64), np.array(ref["sigmas"]))


def test_initialisers_match_the_reference_layer_by_layer(ref):
    """`create_model` draws every tensor from the distribution the reference's constructors use (default_init = variance
    scaling, fan_avg, uniform -- layers.py:54-91; zero-scale Conv_1 / NIN_3 / head; nn.Linear / GroupNorm / bias defaults):
    constant tensors are equal, random ones agree in spread and range (the RNG streams differ: the reference draws and then
    overwrites torch's own Conv3d initialisation)."""
    from helpers import tiny_config
    from meshdiffusion_b200.diffusion.models import utils as mutils
    cfg = tiny_config()
    cfg.device = torch.device("cpu")
    torch.manual_seed(5)
    sd = mutils.create_model(cfg).state_dict()
    theirs = ref["init"]
    assert set(theirs) <= set(sd)
    checked = 0
    for k, r in theirs.items():
        v = sd[k]
        assert v.numel() == r["numel"], k
        if r["const"]:
            assert bool((v == v.flatten()[0]).all()) and abs(float(v.flatten()[0]) - r["mean"]) <= 1e-12, k
            continue
        n = r["numel"]
        tol = max(0.03, 10.0 * (0.2 / n) ** 0.5)
        std = float(v.double().std())
        assert abs(std / r["std"] - 1.0) < tol, (k, std, r["std"])
        if r["absmax"] > 1e-6:  # a uniform law: the sample maximum sits just under the bound in both
            assert abs(float(v.abs().max()) / r["absmax"] - 1.0) < max(0.05, 20.0 / n), (k, float(v.abs().max()), r["absmax"])
        checked += 1
    assert checked > 30

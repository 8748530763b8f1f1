"""CPU: the host loop of the sampler -- every registered predictor / corrector pair, the partial (`cond_gen`) branch with the
reference's (B,B,...) initial-broadcast quirk and `freeze_iters`, and `return_traj` -- is BITWISE equal to the REFERENCE's own
`get_sampling_fn -> pc_sampler` (lib/diffusion/sampling.py:83-132,357-487; its outputs stored in
tests/golden/reference_samplers.npz by oracle/make_host_golden.py) when both drive the stub score model of
oracle/sampler_stub.py with the same seed. (On a CUDA tensor with the native network the configured
ancestral + none pair takes the fused path instead; that path is pinned against reference goldens in tests/test_gpu_sampler.py.)"""
import os

import numpy as np
import pytest
import torch

from helpers import GOLD
from oracle.sampler_stub import VARIANTS, Stub, inputs


@pytest.fixture(scope="module")
def ref():
    return np.load(os.path.join(GOLD, "reference_samplers.npz"))


@pytest.mark.parametrize("variant", VARIANTS, ids=[v[0] for v in VARIANTS])
def test_host_sampler_loop_is_bitwise_the_reference(ref, variant):
    from configs import res64
    from meshdiffusion_b200.diffusion import sampling, sde_lib
    name, pred, corr, nse, pflow, use_partial, freeze, traj, R, iters = variant
    cfg = res64.get_config()
    cfg.device = torch.device("cpu")
    cfg.sampling.method, cfg.sampling.predictor, cfg.sampling.corrector = "pc", pred, corr
    cfg.sampling.n_steps_each, cfg.sampling.probability_flow, cfg.sampling.snr = nse, pflow, 0.16
    if iters is not None:
        cfg.sampling.max_iters = iters
    B = 2
    mask, partial, pmask = inputs(R, B)
    sde = sde_lib.VPSDE(beta_min=cfg.model.beta_min, beta_max=cfg.model.beta_max, N=cfg.model.num_scales, device="cpu")
    fn = sampling.get_sampling_fn(cfg, sde, (B, 4, R, R, R), lambda x: x, 1e-3, grid_mask=mask, return_traj=traj)
    torch.manual_seed(123)
    kw = dict(partial=partial, partial_mask=pmask, partial_channel=0, freeze_iters=freeze) if use_partial else {}
    out, nfe = fn(Stub(), **kw)
    want, want_nfe = torch.from_numpy(ref[name]), int(ref[name + "_nfe"])
    assert nfe == want_nfe
    if traj:
        assert len(out) == len(want) and len(out) > 0
        for a, b in zip(out, want):
            assert torch.equal(a, b)
    else:
        assert out.shape == want.shape and torch.isfinite(want).all()
        assert torch.equal(out, want), f"{name}: max |diff| {(out - want).abs().max().item():.3e}"

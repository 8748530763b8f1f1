"""ORACLE support (test infrastructure only): the stub score model, inputs and variant table with which the reference's
`get_sampling_fn -> pc_sampler` wrote tests/golden/reference_samplers.npz (oracle/make_host_golden.py) and with which
tests/test_sampler_host_parity.py drives this package's sampler host loop."""
import torch


class Stub(torch.nn.Module):
    """Deterministic stand-in for model(x, labels): smooth, label-dependent, mixes neighbouring voxels."""
    def __init__(self):
        super().__init__()
        self.w = torch.nn.Parameter(torch.tensor(0.37))

    def forward(self, x, labels):
        return torch.tanh(self.w * x + 1e-3 * labels.view(-1, 1, 1, 1, 1)) - 0.1 * x.roll(1, 2)


def inputs(R, B):
    g = torch.Generator().manual_seed(77)
    mask = (torch.rand(1, 1, R, R, R, generator=g) < 0.7).float()
    partial = torch.sign(torch.randn(1, 4, R, R, R, generator=g))
    pmask = (torch.rand(1, 4, R, R, R, generator=g) < 0.5).float()
    return mask, partial, pmask


VARIANTS = [  # name, predictor, corrector, n_steps_each, probability_flow, partial, freeze_iters, return_traj, R, iters
    ("ancestral", "ancestral_sampling", "none", 1, False, False, None, False, 8, 25),
    ("em_langevin", "euler_maruyama", "langevin", 2, False, False, None, False, 8, 25),
    ("rd_ald", "reverse_diffusion", "ald", 1, False, False, None, False, 8, 25),
    ("rd_pflow", "reverse_diffusion", "none", 1, True, False, None, False, 8, 25),  # (EM + probability_flow raises in the reference: sampling.py:195)
    ("none_langevin", "none", "langevin", 1, False, False, None, False, 8, 25),
    ("partial", "ancestral_sampling", "none", 1, False, True, 10, False, 8, 25),
    ("partial_all", "reverse_diffusion", "langevin", 1, False, True, None, False, 8, 12),
    ("traj", "ancestral_sampling", "none", 1, False, False, None, True, 4, None),
]

"""Writes the golden files of the CPU tests that compare this package's host-side code with the REFERENCE's own code:

    python oracle/make_host_golden.py      # needs the reference tree (MDB_REFERENCE_DIR)

  tests/golden/reference_host.json.xz             config trees, registries, VP-SDE tables and marginal_prob, EMA recursion,
                                                   optimiser defaults and warm-up, sigmas, per-layer initialiser
                                                   statistics, the checkpoint layout of the reference's model / EMA / Adam,
                                                   and the sha256 of data/tets_to_3dgrid.py::tet_to_grids on the seeded grid
                                                   of the test
  tests/golden/reference_samplers.npz              pc_sampler outputs for the variants of oracle/sampler_stub.py
  tests/golden/reference_checkpoint_tiny.pth.xz   a checkpoint written by the reference's save_checkpoint

Each reference-side piece runs the reference's modules, staged unmodified under baseline/_ref by
baseline/install_reference.py, in a subprocess (through baseline/reference_arm.py), so that its top-level `configs` / `lib`
packages never meet this repository's. The tests read only these files.
"""
import hashlib
import json
import lzma
import os
import shutil
import subprocess
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, ROOT)

# config trees, registries, VP-SDE, EMA, optimiser, sigmas, initialisers (tests/test_reference_host_parity.py)
HOST_SIDE = r'''
import json, sys, torch
root, out = sys.argv[1:3]
sys.path.insert(0, root)
from baseline import reference_arm
ref, config = reference_arm.load("cpu")
import importlib
from configs import res128 as cfg128
import lib.diffusion.losses as rlosses
from lib.diffusion.models.ema import ExponentialMovingAverage

def flat(c, pre=""):
    o = {}
    for k, v in c.items():
        if k == "device":
            continue
        if isinstance(v, dict):
            o.update(flat(v, pre + k + "."))
        else:
            o[pre + k] = list(v) if isinstance(v, tuple) else v
    return o

res = {"res64": flat(config), "res128": flat(cfg128.get_config())}
samp = ref["sampling"]
res["predictors"] = sorted(samp._PREDICTORS)
res["correctors"] = sorted(samp._CORRECTORS)
res["models"] = sorted(ref["mutils"]._MODELS)
sde = ref["sde_lib"].VPSDE(beta_min=config.model.beta_min, beta_max=config.model.beta_max, N=config.model.num_scales)
tables = {n: getattr(sde, n).double().tolist() for n in ("discrete_betas", "alphas", "alphas_cumprod", "sqrt_alphas_cumprod", "sqrt_1m_alphas_cumprod")}
x = torch.linspace(-1, 1, 24).view(2, 3, 4)
t = torch.tensor([0.25, 0.9])
mean, std = sde.marginal_prob(x, t)
tables["mp_mean"], tables["mp_std"] = mean.double().tolist(), std.double().tolist()
res["sde"] = tables
# EMA recursion (ema.py:43-64): three updates of a moving parameter
p = [torch.nn.Parameter(torch.arange(6, dtype=torch.float32))]
ema = ExponentialMovingAverage(p, decay=0.9999)
trace = []
for i in range(3):
    p[0].data.mul_(1.5).add_(0.25)
    ema.update(p)
    trace.append(ema.shadow_params[0].double().tolist())
res["ema"] = trace
# optimiser + optimization_manager on CPU: warm-up lr, clip, one Adam step (losses.py:26-52)
torch.manual_seed(0)
w = [torch.nn.Parameter(torch.randn(5, 3)), torch.nn.Parameter(torch.randn(7))]
opt = rlosses.get_optimizer(config, w)
fn = rlosses.optimization_manager(config)
steps = []
g = torch.Generator().manual_seed(1)
for step in (0, 10, 4999, 20000):
    for q in w:
        q.grad = torch.randn(q.shape, generator=g) * 3.0
    fn(opt, w, step=step)
    steps.append({"lr": opt.param_groups[0]["lr"], "w0": w[0].detach().double().flatten().tolist(), "w1": w[1].detach().double().tolist()})
res["optim"] = {"steps": steps, "defaults": {k: (list(v) if isinstance(v, tuple) else v) for k, v in opt.defaults.items()
                                              if k in ("lr", "betas", "eps", "weight_decay", "amsgrad")}}
res["sigmas"] = [float(v) for v in ref["mutils"].get_sigmas(config)]
# initial weights of a tiny network (the reference's own initialisers): per-tensor statistics
config.data.image_size, config.model.nf, config.model.ch_mult = 16, 32, (1, 2)
config.model.num_res_blocks, config.model.attn_resolutions = 1, (8,)
torch.manual_seed(5)
m = ref["mutils"].create_model(config)
res["init"] = {k: {"std": float(v.double().std()) if v.numel() > 1 else 0.0, "absmax": float(v.abs().max()), "mean": float(v.double().mean()),
                   "numel": v.numel(), "const": bool((v == v.flatten()[0]).all())}
               for k, v in m.state_dict().items() if v.dtype.is_floating_point and k.split(".")[-1] not in ("sigmas", "mask", "coords")}
json.dump(res, open(out, "w"))
print("REF_DONE")
'''

# the host loop of pc_sampler on the stub score model (tests/test_sampler_host_parity.py)
SAMPLER_SIDE = r'''
import sys, torch
root, out = sys.argv[1:3]
sys.path.insert(0, root)
from baseline import reference_arm
ref, config = reference_arm.load("cpu")
from oracle.sampler_stub import Stub, inputs, VARIANTS
sampling, sde_lib = ref["sampling"], ref["sde_lib"]
sde = sde_lib.VPSDE(beta_min=config.model.beta_min, beta_max=config.model.beta_max, N=config.model.num_scales)
res = {}
for name, pred, corr, nse, pflow, use_partial, freeze, traj, R, iters in VARIANTS:
    B = 2
    mask, partial, pmask = inputs(R, B)
    config.sampling.method, config.sampling.predictor, config.sampling.corrector = "pc", pred, corr
    config.sampling.n_steps_each, config.sampling.probability_flow, config.sampling.snr = nse, pflow, 0.16
    fn = sampling.get_sampling_fn(config, sde, (B, 4, R, R, R), lambda x: x, 1e-3, grid_mask=mask, return_traj=traj)
    real = sampling.tqdm.trange
    if iters is not None:
        sampling.tqdm.trange = lambda n, *a, **k: range(min(n, iters))
    try:
        torch.manual_seed(123)
        kw = dict(partial=partial, partial_mask=pmask, partial_channel=0, freeze_iters=freeze) if use_partial else {}
        o, nfe = fn(Stub(), **kw)
    finally:
        sampling.tqdm.trange = real
    res[name] = ([t.clone() for t in o] if traj else o.clone(), nfe)
torch.save(res, out)
print("REF_DONE")
'''

# checkpoints (tests/test_checkpoint_interchange.py): what the reference's restore_checkpoint loads into -- the
# `module.`-prefixed state dict of DDPMRes64 inside nn.DataParallel, the parameter list the positional EMA shadow and the
# Adam state follow, Adam's param groups -- and a checkpoint written by its save_checkpoint after one Adam step and two EMA
# updates
CHECKPOINT_SIDE = r'''
import json, sys, torch
root, layout_out, ckpt_out = sys.argv[1:4]
sys.path.insert(0, root)
from baseline import reference_arm
ref, config = reference_arm.load("cpu")
import lib.diffusion.utils as rutils, lib.diffusion.losses as rlosses
from lib.diffusion.models.ema import ExponentialMovingAverage
config.data.image_size, config.model.nf, config.model.ch_mult = 16, 32, (1, 2)
config.model.num_res_blocks, config.model.attn_resolutions = 1, (8,)

def fresh(seed):
    torch.manual_seed(seed)
    model = ref["mutils"].create_model(config)            # models/utils.py:88-96 -> nn.DataParallel shell, `module.` keys
    ema = ExponentialMovingAverage(model.parameters(), decay=config.model.ema_rate)
    opt = rlosses.get_optimizer(config, model.parameters())
    return dict(optimizer=opt, model=model, ema=ema, step=0)

st = fresh(1)
layout = {"model": [[k, list(v.shape), str(v.dtype)] for k, v in st["model"].state_dict().items()],
          "parameters": [[list(p.shape), p.requires_grad] for p in st["model"].parameters()],
          "param_groups": st["optimizer"].state_dict()["param_groups"], "ema_fields": sorted(st["ema"].state_dict())}
json.dump(layout, open(layout_out, "w"))

st = fresh(2)
# periodic weights and gradients, distinct per tensor: the written file (28 MB) then compresses to a small fixture
for i, p in enumerate(st["model"].parameters()):
    k = torch.arange(p.numel(), dtype=torch.float32).view(p.shape)
    with torch.no_grad():
        p.copy_(((k % 7) - 3) * 1e-2 + 1e-4 * i)
    p.grad = (((k * 5 + i) % 11) - 5) * 1e-3
st["ema"] = ExponentialMovingAverage(st["model"].parameters(), decay=config.model.ema_rate)
st["optimizer"].step()
st["ema"].update(st["model"].parameters())
st["ema"].update(st["model"].parameters())
st["step"] = 11
rutils.save_checkpoint(ckpt_out, st)
print("REF_DONE")
'''


def run_reference_side(program, *args):
    r = subprocess.run([sys.executable, "-c", program, ROOT] + list(args), capture_output=True, text=True, timeout=900,
                       env=dict(os.environ, OMP_NUM_THREADS="4"))
    assert r.returncode == 0 and "REF_DONE" in r.stdout, r.stdout + r.stderr


def tet_to_grids_digest(ref_dir):
    """sha256 of the reference's data/tets_to_3dgrid.py::tet_to_grids on the 64 tet grid with the seeded sdf / deformation
    of tests/test_host.py::test_partial_dmtet_and_grid_producers."""
    from meshdiffusion_b200.geometry import dmtet
    src = open(os.path.join(ref_dir, "data", "tets_to_3dgrid.py")).read().split("if __name__")[0]
    ns = {}
    exec(src, ns)
    verts, _ = dmtet.load_tet_grid(64)
    coords = dmtet.grid_coords_of_tet_vertices(verts)
    g = torch.Generator().manual_seed(3)
    sdf = torch.sign(torch.randn(verts.shape[0], generator=g))
    deform = torch.randn(verts.shape[0], 3, generator=g) * 0.1
    grid = ns["tet_to_grids"](coords, (sdf.unsqueeze(-1), deform), 64)
    return hashlib.sha256(grid.contiguous().numpy().tobytes()).hexdigest()


def main():
    from baseline import install_reference
    if install_reference.install() is None:
        raise SystemExit(f"the reference tree is not at {install_reference.REF} (set MDB_REFERENCE_DIR)")
    with tempfile.TemporaryDirectory() as tmp:
        run_reference_side(HOST_SIDE, os.path.join(tmp, "host.json"))
        host = json.load(open(os.path.join(tmp, "host.json")))
        run_reference_side(CHECKPOINT_SIDE, os.path.join(tmp, "layout.json"), os.path.join(tmp, "ckpt.pth"))
        host["checkpoint_layout"] = json.load(open(os.path.join(tmp, "layout.json")))
        with open(os.path.join(tmp, "ckpt.pth"), "rb") as src, \
                lzma.open(os.path.join(GOLD, "reference_checkpoint_tiny.pth.xz"), "wb", preset=9 | lzma.PRESET_EXTREME) as dst:
            shutil.copyfileobj(src, dst)
        host["tet_to_grids_sha256"] = tet_to_grids_digest(install_reference.REF)
        with lzma.open(os.path.join(GOLD, "reference_host.json.xz"), "wt", preset=9) as f:
            json.dump(host, f)
        run_reference_side(SAMPLER_SIDE, os.path.join(tmp, "samplers.pt"))
        samplers = torch.load(os.path.join(tmp, "samplers.pt"), weights_only=False)
    arrays = {}
    for name, (out, nfe) in samplers.items():
        arrays[name] = (torch.stack(out) if isinstance(out, list) else out).numpy()
        arrays[name + "_nfe"] = np.array(nfe, np.int64)
    np.savez_compressed(os.path.join(GOLD, "reference_samplers.npz"), **arrays)
    for n in ("reference_host.json.xz", "reference_checkpoint_tiny.pth.xz", "reference_samplers.npz"):
        print(n, os.path.getsize(os.path.join(GOLD, n)), "bytes")


if __name__ == "__main__":
    main()

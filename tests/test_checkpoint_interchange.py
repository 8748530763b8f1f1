"""CPU: checkpoints interchange with the REFERENCE's own code in both directions (the drop-in contract of SURVEY 8b:
`torch.save({'optimizer','model','ema','step'})` with `module.`-prefixed model keys, positional EMA shadow list, the stock
Adam state). oracle/make_host_golden.py stores, from the reference's code, what its `lib.diffusion.utils.restore_checkpoint`
loads into -- the state dict of `DDPMRes64` inside `nn.DataParallel`, the parameter list that `ExponentialMovingAverage`
and `losses.get_optimizer`'s Adam follow (tests/golden/reference_host.json.xz) -- and a checkpoint its `save_checkpoint` wrote
(tests/golden/reference_checkpoint_tiny.pth.xz)."""
import json
import lzma
import os
import shutil

import torch

from helpers import GOLD, tiny_config


def _restore_as_the_reference(path, layout):
    """What the reference's restore_checkpoint (utils.py:6-20) does with `path` on CPU, over a state of its layout:
    torch.load, Adam.load_state_dict, model.load_state_dict(strict=False), EMA.load_state_dict (attribute copy)."""
    loaded = torch.load(path, map_location="cpu")
    assert {"optimizer", "model", "ema", "step"} <= set(loaded)
    model = {k: (shape, dtype) for k, shape, dtype in layout["model"]}
    for k, v in loaded["model"].items():  # strict=False skips unknown keys, but a shape mismatch still raises
        if k in model:
            assert list(v.shape) == model[k][0], (k, list(v.shape), model[k][0])
    params = [torch.nn.Parameter(torch.zeros(shape), requires_grad=rg) for shape, rg in layout["parameters"]]
    hyper = {k: (tuple(v) if isinstance(v, list) else v) for k, v in layout["param_groups"][0].items() if k != "params"}
    opt = torch.optim.Adam(params, **hyper)
    opt.load_state_dict(loaded["optimizer"])
    assert set(layout["ema_fields"]) <= set(loaded["ema"])
    shadow = loaded["ema"]["shadow_params"]
    assert [list(t.shape) for t in shadow] == [shape for shape, rg in layout["parameters"] if rg]
    return loaded, model, opt, params


def test_checkpoints_interchange_with_the_reference_code(tmp_path):
    from meshdiffusion_b200.diffusion import losses
    from meshdiffusion_b200.diffusion.models import utils as mutils
    from meshdiffusion_b200.diffusion.models.ema import ExponentialMovingAverage
    from meshdiffusion_b200.diffusion.utils import restore_checkpoint, save_checkpoint

    cfg = tiny_config()
    cfg.device = torch.device("cpu")

    def fresh(seed):
        torch.manual_seed(seed)
        model = mutils.create_model(cfg)
        return dict(optimizer=losses.get_optimizer(cfg, model.parameters()), model=model,
                    ema=ExponentialMovingAverage(model.parameters(), decay=cfg.model.ema_rate), step=0)

    # ---- ours -> file. The fused optimiser step needs the GPU, so its (stock Adam) state is filled in by hand.
    st = fresh(5)
    g = torch.Generator().manual_seed(6)
    with torch.no_grad():
        for p in st["model"].parameters():
            p.add_(torch.randn(p.shape, generator=g) * 1e-2)
    opt = st["optimizer"]
    for p in st["model"].parameters():
        if p.requires_grad:
            opt.state[p] = {"step": torch.tensor(3.0), "exp_avg": torch.randn(p.shape, generator=g),
                            "exp_avg_sq": torch.rand(p.shape, generator=g)}
    st["ema"].update(st["model"].parameters())
    st["step"] = 7
    ours_ckpt = str(tmp_path / "ours.pth")
    save_checkpoint(ours_ckpt, st)
    plain = {"model": {k: v.clone() for k, v in st["model"].state_dict().items()},
             "ema_shadow": [t.clone() for t in st["ema"].shadow_params], "ema_num_updates": st["ema"].num_updates,
             "ema_decay": st["ema"].decay,
             "opt_state": {i: {k: v.clone() for k, v in s.items()} for i, s in opt.state_dict()["state"].items()}}

    # ---- the file -> the reference's restore_checkpoint
    layout = json.load(lzma.open(os.path.join(GOLD, "reference_host.json.xz"), "rt"))["checkpoint_layout"]
    loaded, model, ropt, rparams = _restore_as_the_reference(ours_ckpt, layout)
    assert loaded["step"] == 7
    assert set(model) == set(plain["model"]), set(model) ^ set(plain["model"])
    for k, v in plain["model"].items():
        assert model[k][1] == str(v.dtype) and torch.equal(loaded["model"][k], v), k
    assert loaded["ema"]["num_updates"] == plain["ema_num_updates"] and loaded["ema"]["decay"] == plain["ema_decay"]
    for a, b in zip(loaded["ema"]["shadow_params"], plain["ema_shadow"]):
        assert torch.equal(a, b)
    ost = ropt.state_dict()
    assert len(ost["state"]) == len(plain["opt_state"])
    for i, s in plain["opt_state"].items():
        for f in ("exp_avg", "exp_avg_sq"):
            assert torch.equal(ost["state"][i][f], s[f]), (i, f)
        assert float(ost["state"][i]["step"]) == float(s["step"])
    # the restored reference optimiser keeps stepping (its state is the stock Adam layout)
    for p in rparams:
        p.grad = torch.zeros_like(p)
    ropt.step()

    # ---- the reference's file -> ours
    ref_ckpt = str(tmp_path / "ref.pth")
    with lzma.open(os.path.join(GOLD, "reference_checkpoint_tiny.pth.xz"), "rb") as src, open(ref_ckpt, "wb") as dst:
        shutil.copyfileobj(src, dst)
    raw = torch.load(ref_ckpt, map_location="cpu")
    plain = {"model": raw["model"], "ema_shadow": raw["ema"]["shadow_params"], "ema_num_updates": raw["ema"]["num_updates"],
             "opt_state": raw["optimizer"]["state"], "param_groups": raw["optimizer"]["param_groups"]}
    st2 = restore_checkpoint(ref_ckpt, fresh(8), "cpu")
    assert st2["step"] == 11
    sd = st2["model"].state_dict()
    assert set(sd) == set(plain["model"])
    for k, v in plain["model"].items():
        assert sd[k].dtype == v.dtype and torch.equal(sd[k], v), k
    assert st2["ema"].num_updates == plain["ema_num_updates"] == 2
    for a, b in zip(st2["ema"].shadow_params, plain["ema_shadow"]):
        assert torch.equal(a, b)
    ost = st2["optimizer"].state_dict()
    assert set(ost["state"]) == set(plain["opt_state"])
    for i, s in plain["opt_state"].items():
        for f in ("exp_avg", "exp_avg_sq"):
            assert torch.equal(ost["state"][i][f], s[f]), (i, f)
        assert float(ost["state"][i]["step"]) == float(s["step"]) == 1.0
    for ga, gb in zip(ost["param_groups"], plain["param_groups"]):
        for key in ("lr", "betas", "eps", "weight_decay"):
            assert ga[key] == gb[key], key
        assert ga["params"] == gb["params"]

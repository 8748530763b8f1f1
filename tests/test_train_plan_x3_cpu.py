"""Host-side checks of the split-bf16 ("bf16x3") training plan and its configuration key, built GPU-less through
mdb_unet_create_dry."""
import ctypes

import pytest

from helpers import full_config, tiny_config


def _dry(cfg, batch, precision):
    """(arena bytes, [(name, shape)]) of a dry training plan."""
    from meshdiffusion_b200 import _native
    from meshdiffusion_b200.diffusion.models import ddpm
    L = _native.lib()
    c = ddpm._config_c(ddpm.arch_from_config(cfg), batch, precision, training=True)
    h = ctypes.c_void_p()
    _native.check(L.mdb_unet_create_dry(ctypes.byref(c), ctypes.byref(h)))
    try:
        arena = ctypes.c_longlong()
        _native.check(L.mdb_unet_info(h, None, ctypes.byref(arena), None, None))
        table = []
        for i in range(L.mdb_unet_num_params(h)):
            name, numel, nd = ctypes.c_char_p(), ctypes.c_longlong(), ctypes.c_int()
            shape = (ctypes.c_longlong * 8)()
            _native.check(L.mdb_unet_param_info(h, i, ctypes.byref(name), ctypes.byref(numel), ctypes.byref(nd), shape))
            table.append((name.value.decode(), tuple(int(shape[j]) for j in range(nd.value))))
        return arena.value, table
    finally:
        L.mdb_unet_destroy(h)


@pytest.mark.parametrize("name,batch", [("tiny", 3), ("res64", 1), ("res128", 1)])
def test_x3_training_plan_builds_frees_everything_and_keeps_the_param_table(name, batch):
    """The builder throws if any block stays in the arena after the backward emitters ran. Split-bf16 activations and
    gradients take twice the bytes of bf16 ones, fp32 scratch (split-K partials, attention logits, GroupNorm partials)
    does not grow: the arena lies between 1x and 2.2x the bf16 training arena."""
    cfg = tiny_config("res64", "bf16") if name == "tiny" else full_config(name, "bf16")
    a_bf16, t_bf16 = _dry(cfg, batch, "bf16")
    a_x3, t_x3 = _dry(cfg, batch, "bf16x3")
    assert t_x3 == t_bf16
    ratio = a_x3 / a_bf16
    print(f"{name} B{batch}: training arena bf16 {a_bf16 / 2**20:.1f} MiB, bf16x3 {a_x3 / 2**20:.1f} MiB, ratio {ratio:.3f}")
    assert 1.0 < ratio <= 2.2


def test_config_c_carries_the_x3_training_precision():
    from meshdiffusion_b200.diffusion.models import ddpm
    c = ddpm._config_c(ddpm.arch_from_config(tiny_config("res64", "bf16")), 2, "bf16x3", training=True)
    assert c.precision == 2 and c.training == 1


def test_training_compute_dtype_defaults_to_bf16():
    from configs import default_configs, res64, res128
    assert default_configs.get_default_configs().training.compute_dtype == "bf16"
    assert res64.get_config().training.compute_dtype == "bf16"
    assert res128.get_config().training.compute_dtype == "bf16"


@pytest.mark.parametrize("value", ["tf32", "fp32", "bf16X3", ""])
def test_unknown_training_compute_dtype_is_refused_at_construction(value):
    from meshdiffusion_b200.diffusion.models import ddpm
    cfg = tiny_config("res64", "bf16")
    cfg.training.compute_dtype = value
    with pytest.raises(ValueError, match="training.compute_dtype"):
        ddpm.DDPMRes64(cfg)


def test_x3_training_mode_is_read_from_the_config():
    from meshdiffusion_b200.diffusion.models import ddpm
    cfg = tiny_config("res64", "bf16")
    assert ddpm.DDPMRes64(cfg).train_precision == "bf16"
    cfg.training.compute_dtype = "bf16x3"
    assert ddpm.DDPMRes64(cfg).train_precision == "bf16x3"

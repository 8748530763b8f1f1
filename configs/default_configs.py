"""Default configuration tree (same keys and values as the reference's configs/default_configs.py:5-89)."""
import torch

from meshdiffusion_b200.compat.install import ensure_ml_collections

ensure_ml_collections()
import ml_collections  # noqa: E402

_DEFAULTS = {
    "training": dict(batch_size=64, n_iters=2400001, snapshot_freq=50000, log_freq=50, eval_freq=100,
                     snapshot_freq_for_preemption=5000, snapshot_sampling=True, likelihood_weighting=False,
                     continuous=True, reduce_mean=False, iter_size=1, loss_type="l2", train_dir="PLACEHOLDER",
                     # engine knob (not a reference key): training operand mode, 'bf16' or 'bf16x3' (split bf16, fp32-class
                     # gradients at about a third of the tensor rate)
                     compute_dtype="bf16"),
    "sampling": dict(n_steps_each=1, noise_removal=True, probability_flow=False, snr=0.075),
    "eval": dict(begin_ckpt=50, end_ckpt=96, batch_size=512, enable_sampling=True, num_samples=50000, enable_loss=True,
                 enable_bpd=False, bpd_dataset="test", ckpt_path="PLACEHOLDER", partial_dmtet_path="PLACEHOLDER",
                 tet_path="PLACEHOLDER", freeze_iters=950),
    "data": dict(dataset="LSUN", image_size=256, random_flip=True, uniform_dequantization=False, centered=False,
                 num_channels=3, num_workers=4, normalize_sdf=True, meta_path="PLACEHOLDER",
                 filter_meta_path="PLACEHOLDER", extension="pt"),
    "model": dict(sigma_max=378, sigma_min=0.01, num_scales=2000, beta_min=0.1, beta_max=20.0, dropout=0.0,
                  embedding_type="fourier", deform_scale=1.0),
    "optim": dict(weight_decay=0, optimizer="Adam", lr=2e-4, beta1=0.9, eps=1e-8, warmup=5000, grad_clip=1.0),
    "render": dict(),
}


def get_default_configs():
    config = ml_collections.ConfigDict()
    for section, values in _DEFAULTS.items():
        config[section] = ml_collections.ConfigDict(dict(values))
    config.seed = 42
    config.device = torch.device("cuda:0") if torch.cuda.is_available() else torch.device("cpu")
    return config

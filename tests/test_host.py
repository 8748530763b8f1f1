"""CPU: host-side logic -- parameter table vs the reference's state_dict, checkpoint layout, config surface, CLI,
registries, EMA arithmetic, and a world_size-2 gloo run of the batch-sharded sampler plumbing."""
import hashlib
import json
import lzma
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from helpers import GOLD, ROOT, full_config, tiny_config


@pytest.mark.parametrize("name", ["res64", "res128"])
def test_state_dict_matches_reference_layout(name):
    """Keys (with the DataParallel 'module.' prefix), order, shapes and dtypes of the reference's state_dict, and the
    order of trainable parameters that the positional EMA list depends on (golden from the reference constructor)."""
    from meshdiffusion_b200.diffusion.models import utils as mutils
    gold = json.load(open(os.path.join(GOLD, "param_tables.json")))[name]
    cfg = full_config(name)
    cfg.device = torch.device("cpu")
    with torch.device("meta"):
        pass
    model = mutils.create_model(cfg)
    sd = model.state_dict()
    ours = {k: (list(v.shape), str(v.dtype)) for k, v in sd.items()}
    ref = {k: (shape, dt) for k, shape, dt in gold["state_dict"]}
    assert set(ours) == set(ref), (sorted(set(ref) - set(ours))[:5], sorted(set(ours) - set(ref))[:5])
    for k in ref:
        assert ours[k] == ref[k], (k, ours[k], ref[k])
    trainable = [n for n, p in model.named_parameters() if p.requires_grad]
    assert trainable == gold["trainable"]


def test_checkpoint_roundtrip(tmp_path):
    from meshdiffusion_b200.diffusion import losses
    from meshdiffusion_b200.diffusion.models import utils as mutils
    from meshdiffusion_b200.diffusion.models.ema import ExponentialMovingAverage
    from meshdiffusion_b200.diffusion.utils import restore_checkpoint, save_checkpoint
    cfg = tiny_config()
    cfg.device = torch.device("cpu")
    model = mutils.create_model(cfg)
    opt = losses.get_optimizer(cfg, model.parameters())
    ema = ExponentialMovingAverage(model.parameters(), decay=cfg.model.ema_rate)
    ema.update(model.parameters())
    state = dict(optimizer=opt, model=model, ema=ema, step=7)
    path = os.path.join(tmp_path, "checkpoints-meta", "checkpoint.pth")
    save_checkpoint(path, state)
    raw = torch.load(path, map_location="cpu", weights_only=False)
    assert set(raw) == {"optimizer", "model", "ema", "step"} and raw["step"] == 7
    assert all(k.startswith("module.") for k in raw["model"])
    assert set(raw["ema"]) == {"decay", "num_updates", "shadow_params"} and raw["ema"]["num_updates"] == 1
    model2 = mutils.create_model(cfg)
    state2 = dict(optimizer=losses.get_optimizer(cfg, model2.parameters()), model=model2,
                  ema=ExponentialMovingAverage(model2.parameters(), decay=0.5), step=0)
    state2 = restore_checkpoint(path, state2, device="cpu")
    assert state2["step"] == 7 and state2["ema"].decay == cfg.model.ema_rate
    for (k, a), (_, b) in zip(model.state_dict().items(), model2.state_dict().items()):
        assert torch.equal(a, b), k
    # missing file: warning + unchanged state (lib/diffusion/utils.py:7-13)
    assert restore_checkpoint(os.path.join(tmp_path, "nope", "x.pth"), state2, "cpu")["step"] == 7


def test_ema_arithmetic():
    from meshdiffusion_b200.diffusion.models.ema import ExponentialMovingAverage
    p = [torch.nn.Parameter(torch.ones(4)), torch.nn.Parameter(torch.zeros(3), requires_grad=False)]
    ema = ExponentialMovingAverage(p, decay=0.9999)
    assert len(ema.shadow_params) == 1
    p[0].data.fill_(3.0)
    ema.update(p)  # decay_t = min(0.9999, 2/11)
    d = 2.0 / 11.0
    assert torch.allclose(ema.shadow_params[0], torch.full((4,), 1.0 - (1 - d) * (1.0 - 3.0)))


def test_config_surface_and_cli_overrides():
    import main_diffusion
    path, mode, ov = main_diffusion.parse_args(["--config=configs/res64.py", "--mode=uncond_gen", "--config.eval.batch_size=7",
                                                "--config.eval.eval_dir=/tmp/x", "--config.new.key=(1,2)"])
    assert mode == "uncond_gen" and ("eval.batch_size", 7) in ov and ("new.key", (1, 2)) in ov
    cfg = main_diffusion.load_config_file(os.path.join(ROOT, path))
    for k, v in ov:
        cfg.set_by_path(k, v)
    assert cfg.eval.batch_size == 7 and cfg.new.key == (1, 2) and cfg.eval.eval_dir == "/tmp/x"
    assert cfg.model.ch_mult == (1, 1, 2, 4, 4) and cfg.sampling.predictor == "ancestral_sampling" and cfg.optim.lr == 2e-5
    with pytest.raises(SystemExit):
        main_diffusion.parse_args(["--config=c.py", "--mode=bogus"])


def test_registries():
    from meshdiffusion_b200.diffusion import sampling
    from meshdiffusion_b200.diffusion.models import ddpm, utils as mutils
    assert mutils.get_model("ddpm_res64") is ddpm.DDPMRes64
    assert mutils.get_model("ddpm_res128_v2") is mutils.get_model("ddpm_res128")
    for n in ("euler_maruyama", "reverse_diffusion", "ancestral_sampling", "none"):
        assert sampling.get_predictor(n)
    for n in ("langevin", "ald", "none"):
        assert sampling.get_corrector(n)
    with pytest.raises(ValueError):
        mutils.register_model(ddpm.DDPMRes64, name="ddpm_res64")


def test_score_net_refuses_cpu():
    from meshdiffusion_b200 import _native
    from meshdiffusion_b200.diffusion.models import utils as mutils
    cfg = tiny_config()
    cfg.device = torch.device("cpu")
    model = mutils.create_model(cfg)
    with pytest.raises(_native.NativeError):
        model(torch.zeros(1, 4, 16, 16, 16), torch.zeros(1))


GLOO_CHILD = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, %r)
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
# the sampler shards the batch with no data-path collective: only timing / bookkeeping crosses ranks
from meshdiffusion_b200.diffusion import sde_lib
sde = sde_lib.VPSDE(device="cpu")
torch.manual_seed(42 + rank)
x = torch.randn(2, 4, 8, 8, 8)
t = torch.tensor([float(rank + 1)])
dist.all_reduce(t, op=dist.ReduceOp.MAX)
gathered = [torch.zeros(2, 4, 8, 8, 8) for _ in range(world)]
dist.all_gather(gathered, x)
assert t.item() == world and not torch.equal(gathered[0], gathered[1])
print("RANK_OK", rank, float(sde.discrete_betas[0]))
dist.destroy_process_group()
''' % ROOT


def test_world_size_2_gloo_plumbing(tmp_path):
    script = os.path.join(tmp_path, "child.py")
    open(script, "w").write(GLOO_CHILD)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29533", script],
                       capture_output=True, text=True, timeout=240)
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.count("RANK_OK") == 2


GLOO_TRAIN_CHILD = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, %r)
sys.path.insert(0, os.path.join(%r, "tests"))
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
from helpers import tiny_config
from meshdiffusion_b200.diffusion.models import utils as mutils
cfg = tiny_config("res64", "bf16")
cfg.device = torch.device("cpu")
net = mutils.create_model(cfg, use_parallel=False)
# data-parallel training exchanges ONE buffer: the flat fp32 gradient the engine writes (here filled by hand: the
# engine itself needs a GPU); every p.grad is a view of it, so the optimiser sees the averaged gradient
n = sum(p.numel() for p in net.parameters())
net._flat_grad = torch.full((n,), float(rank + 1))
view = net._flat_grad[:10]
net.allreduce_grads()
assert torch.allclose(net._flat_grad, torch.full((n,), (1 + world) / 2.0)), net._flat_grad[:4]
assert view.data_ptr() == net._flat_grad.data_ptr() and float(view[0]) == (1 + world) / 2.0
print("TRAIN_RANK_OK", rank)
dist.destroy_process_group()
''' % (ROOT, ROOT)


def test_world_size_2_gradient_allreduce(tmp_path):
    script = os.path.join(tmp_path, "child_train.py")
    open(script, "w").write(GLOO_TRAIN_CHILD)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29534", script],
                       capture_output=True, text=True, timeout=240)
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.count("TRAIN_RANK_OK") == 2


GLOO_BUCKET_CHILD = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, %r)
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
from meshdiffusion_b200.diffusion.models.ddpm import make_grad_buckets
# a flat gradient buffer laid out like the engine's: slots in forward order, readiness falling with the offset, one
# late-ready slot at the front (the time-embedding MLP) and a never-written slot (ready 0) in the middle
g = torch.Generator().manual_seed(7)
numels = [int(v) for v in torch.randint(1, 5000, (60,), generator=g)]
offs = [0]
for n in numels[:-1]:
    offs.append(offs[-1] + n)
total = offs[-1] + numels[-1]
ready = [300] + [290 - 4 * i for i in range(59)]
ready[20] = 0
buckets = make_grad_buckets(list(zip(offs, numels, ready)), total, 16000 * 4)
# the ranges tile the buffer exactly, each at least one bucket size (except the remainder at the front)
cover = sorted((lo, hi) for _, lo, hi in buckets)
assert cover[0][0] == 0 and cover[-1][1] == total and all(a[1] == b[0] for a, b in zip(cover, cover[1:])), cover
assert len(buckets) >= 4 and all(hi - lo >= 16000 for _, lo, hi in buckets if lo != 0)
assert [b[0] for b in buckets] == sorted(b[0] for b in buckets)
for rdy, lo, hi in buckets:  # a range is ready only when all of its slots are
    assert rdy == max(r for o, n, r in zip(offs, numels, ready) if lo <= o < hi)
assert buckets[-1][1] == 0 and buckets[-1][0] == 300  # the front range (late slot) goes last
# bucket-by-bucket mean == whole-buffer mean
flat = torch.randn(total, generator=torch.Generator().manual_seed(rank))
whole = flat.clone()
dist.all_reduce(whole); whole /= world
for _, lo, hi in buckets:
    dist.all_reduce(flat[lo:hi])
flat /= world
assert torch.equal(flat, whole)
print("BUCKET_RANK_OK", rank)
dist.destroy_process_group()
''' % ROOT


def test_world_size_2_bucketed_gradient_mean(tmp_path):
    """The data-parallel exchange's host logic on CPU/gloo: make_grad_buckets tiles the flat buffer from its end in
    readiness order, and reducing it bucket by bucket equals reducing it whole."""
    script = os.path.join(tmp_path, "child_buckets.py")
    open(script, "w").write(GLOO_BUCKET_CHILD)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                        "--master-addr", "127.0.0.1", "--master-port", "29535", script],
                       capture_output=True, text=True, timeout=240)
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.count("BUCKET_RANK_OK") == 2


def test_dataset_items_match_reference_golden(tmp_path):
    """ShapeNetDMTetDataset: items bit-identical to the reference class on the committed synthetic shapes (filter list,
    sign quirk, seeded jitter augmentation, mask multiply, right padding); golden from the reference class itself."""
    from meshdiffusion_b200.dataset.shapenet_dmtet_dataset import ShapeNetDMTetDataset
    gold = np.load(os.path.join(GOLD, "dataset_items.npz"))
    paths = []
    for i, raw in enumerate(gold["raw"]):
        p = os.path.join(tmp_path, f"shape_{i}.pt")
        torch.save(torch.tensor(raw), p)
        paths.append(p)
    meta = os.path.join(tmp_path, "meta.json")
    json.dump(paths, open(meta, "w"))
    filt = os.path.join(tmp_path, "filter.json")
    json.dump([int(v) for v in gold["filter"]], open(filt, "w"))
    mask = torch.tensor(gold["mask"])
    k = 0
    for aug in (False, True):
        ds = ShapeNetDMTetDataset(meta, mask, deform_scale=3.0, aug=aug, filter_meta_path=filt, normalize_sdf=True, extension="pt")
        assert len(ds) == 3
        for i in range(3):
            torch.manual_seed(100 + i)
            assert np.array_equal(ds[i].numpy(), gold["items"][k]), (aug, i)
            k += 1
    # the .npy branch (a NameError in the reference) loads the same values
    np.save(os.path.join(tmp_path, "shape_9.npy"), gold["raw"][0])
    json.dump([os.path.join(tmp_path, "shape_9.npy")], open(meta, "w"))
    ds = ShapeNetDMTetDataset(meta, mask, aug=False, extension="npy")
    assert np.array_equal(ds[0].numpy(), gold["items"][0])


def test_on_device_augmentation_matches_items(tmp_path):
    """augment_on_device (the batched form of the loader's aug pipeline) == the reference golden items when it is handed the
    same per-item jitter draws."""
    from meshdiffusion_b200.dataset.shapenet_dmtet_dataset import augment_on_device
    gold = np.load(os.path.join(GOLD, "dataset_items.npz"))
    keep = [i for i in range(len(gold["raw"])) if i in set(int(v) for v in gold["filter"])]
    raw = torch.tensor(gold["raw"][keep])
    shifts = []
    for i in range(len(keep)):
        torch.manual_seed(100 + i)
        shifts.append(torch.rand(3))
    out = augment_on_device(raw, torch.tensor(gold["mask"]), torch.stack(shifts))
    assert np.array_equal(out.numpy(), gold["items"][len(keep):]), "batched augmentation differs from the reference items"


def test_partial_dmtet_and_grid_producers():
    """geometry/formats.py against the reference's own code: data/tets_to_3dgrid.py::tet_to_grids (its output pinned by a
    digest), and the fit_singleview.py:798-827 visibility tail restated literally."""
    from meshdiffusion_b200.geometry import dmtet, formats
    verts, idx = dmtet.load_tet_grid(64)
    coords = dmtet.grid_coords_of_tet_vertices(verts)
    g = torch.Generator().manual_seed(3)
    Nv, Fn = verts.shape[0], idx.shape[0]
    sdf = torch.sign(torch.randn(Nv, generator=g))
    deform = torch.randn(Nv, 3, generator=g) * 0.1
    grid = formats.tets_to_3dgrid(coords, sdf, deform, 64)
    assert grid.shape == (4, 64, 64, 64)
    x, y, z = coords[:, 0], coords[:, 1], coords[:, 2]
    assert torch.equal(grid[0, x, y, z], sdf) and torch.equal(grid[1:, x, y, z], deform.t())
    assert torch.equal(grid.abs().sum(0) != 0, dmtet.grid_mask_from_tets(64) == 1)  # sdf is +-1 on every tet vertex
    # the reference function itself on the same inputs, as its sha256 (oracle/make_host_golden.py)
    want = json.load(lzma.open(os.path.join(GOLD, "reference_host.json.xz"), "rt"))["tet_to_grids_sha256"]
    assert hashlib.sha256(grid.contiguous().numpy().tobytes()).hexdigest() == want
    # visibility -> dmtet.pt
    vis_id = torch.randperm(Fn, generator=g)[:5000]
    rast_id = torch.randperm(Fn, generator=g)[:300]
    d = formats.partial_dmtet_from_visibility(torch.tensor(idx), Nv, sdf, deform, vis_id, rast_id)
    assert set(d) == {"sdf", "deform", "vis", "vis_rast"} and d["vis"].dtype == torch.float32 and d["vis_rast"].dtype == torch.bool
    tets = torch.tensor(idx).long()
    visible = torch.zeros(Fn)
    visible[vis_id] = 1
    both = visible.clone()
    both[rast_id.unique()] = 1
    want_vis = torch.zeros(Nv)
    want_vis[tets[visible == 1].unique()] = 1
    want_vr = want_vis.clone()
    want_vr[tets[both == 1].unique()] = 1
    assert torch.equal(d["vis"], want_vis) and torch.equal(d["vis_rast"], want_vr.bool())
    assert d["vis_rast"].sum() >= d["vis"].sum() > 0


def test_statistics_record_round_trip():
    """The split fixed-point (lo, hi) GroupNorm statistics record (csrc/gn_stats.cuh) as the Python mirror encodes it:
    exact round trip over 20 orders of magnitude, lo within +-2^15 * 2^24, far beyond the 5.5e11 single-word range."""
    from meshdiffusion_b200 import ops
    v = torch.tensor([[[0.0, 1.5], [-3.25e-5, 7.0e-6], [1234.5, 5.5e11], [-9.87e8, 4.3e12], [3.0e15, 1.0e19]]], dtype=torch.float64)
    w = ops.stats_to_words(v)
    assert w.dtype == torch.int64 and w.shape == (1, 5, ops.STAT_WORDS)
    assert (w[..., 0].abs() <= 2 ** 39).all() and (w[..., 2].abs() <= 2 ** 39).all()
    back = ops.words_to_stats(w)
    assert torch.allclose(back, v, rtol=1e-12, atol=2 ** -25)
    # sums of many records stay exact in integer arithmetic (what the kernels' atomics do)
    many = ops.stats_to_words(torch.full((1, 1, 2), 40000.123, dtype=torch.float64)).repeat(1, 1000, 1).sum(dim=1, keepdim=True)
    assert torch.allclose(ops.words_to_stats(many), torch.full((1, 1, 2), 40000.123 * 1000, dtype=torch.float64), rtol=1e-9)


def test_trainer_loop_bounds_checkpoint_names_and_resume(tmp_path, monkeypatch):
    """The host loop of `--mode=train` with a stubbed optimiser step (the real one needs the GPU): iterations
    range(initial_step // iter_size, n_iters + 1), flags (clear_grad on the first, update_param on the last micro-batch),
    `checkpoint_<step>.pth` every snapshot_freq AND at step == n_iters, the pre-emption file every
    snapshot_freq_for_preemption, and auto-resume from it -- the reference's trainer.py:44-51,95-130."""
    from meshdiffusion_b200.diffusion import trainer
    cfg = tiny_config()
    cfg.device = torch.device("cpu")
    cfg.data.synthetic = True
    cfg.training.train_dir = str(tmp_path / "run")
    cfg.training.n_iters, cfg.training.iter_size, cfg.training.batch_size = 5, 2, 2
    cfg.training.snapshot_freq, cfg.training.snapshot_freq_for_preemption, cfg.training.log_freq = 2, 3, 1
    R = cfg.data.image_size
    monkeypatch.setattr(trainer, "load_grid_mask", lambda r, dev: torch.ones(r, r, r))
    monkeypatch.setattr(trainer, "synthetic_grids", lambda b, r, dev, gen=None: torch.zeros(b, 4, r, r, r))
    calls = []

    def fake_make_train_step(config, state, sde, mask):
        def step_fn(state, batch, clear_grad=True, update_param=True):
            assert tuple(batch.shape) == (2, 4, R, R, R)
            calls.append((int(state["step"]), clear_grad, update_param))
            state["step"] += 1  # losses.py:128 of the reference: the counter advances every micro-step
            return {"loss": torch.tensor(1.0)}
        return step_fn

    monkeypatch.setattr(trainer, "make_train_step", fake_make_train_step)
    trainer.train(cfg)
    ck = os.path.join(cfg.training.train_dir, "checkpoints")
    assert sorted(os.listdir(ck)) == ["checkpoint_2.pth", "checkpoint_4.pth", "checkpoint_5.pth"]
    meta = os.path.join(cfg.training.train_dir, "checkpoints-meta", "checkpoint.pth")
    assert os.path.exists(meta)
    assert len(calls) == 6 * 2 and [c[1:] for c in calls[:2]] == [(True, False), (False, True)]
    assert torch.load(os.path.join(ck, "checkpoint_5.pth"), weights_only=False)["step"] == 12
    assert torch.load(meta, weights_only=False)["step"] == 8  # written after iteration 3 (4 iterations x 2 micro-steps)
    # resume: the pre-emption file holds step 8 -> the loop restarts at iteration 8 // 2 = 4
    calls.clear()
    cfg.training.n_iters = 6
    trainer.train(cfg)
    assert [c[0] for c in calls] == [8, 9, 10, 11, 12, 13]
    assert "checkpoint_6.pth" in os.listdir(ck)

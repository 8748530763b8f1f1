"""Training-step throughput of the PRODUCT training path (BASELINE.json configs[2]: res64 train, synthetic 4x64^3 grids,
bf16 operands, fp32 master weights + Adam + EMA, data-parallel gradient mean).

    python tools/bench_train.py [--batch 16] [--iters 4] [--steps 3] [--warmup 1] [--precision bf16|bf16x3]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P tools/bench_train.py ...

The step that is timed is the one `main_diffusion.py --mode=train` runs: trainer.build_state / trainer.make_train_step ->
losses.get_step_fn (native perturb + loss node, engine forward / backward through loss.backward(), bucketed all-reduce
overlapped with the backward pass, FusedAdam with clip coefficient + EMA in one pass). One optimiser step = `iters`
micro-batches of `batch` grids per GPU. Prints ONE JSON line: samples/s over all ranks, the device-time split (CUDA events
around the product methods; `allreduce` is the EXPOSED wait of the optimiser on the side-stream reductions) and the achieved
tensor-core rate (forward + backward GEMM FLOPs / their device time) against the measured sustained bf16 peak (divided by
the 3 MMAs per product in the split-bf16 mode, `--precision bf16x3`, as bench.py does), and the engine's arena size.
"""
import argparse
import ctypes
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ.setdefault("NCCL_DEBUG", "WARN")

import torch  # noqa: E402


MMA_PER_PRODUCT = {"bf16": 1.0, "bf16x3": 3.0}


def run(batch=16, iters=4, steps=3, warmup=1, config="res64", dropout=0.1, no_overlap=False, profile=None, precision="bf16"):
    """Runs the measurement on every rank (joins the NCCL group if the caller has not) and returns the JSON line as a dict
    on rank 0 (None elsewhere). bench.py calls this in-process for its `train` leg. `precision`: the training operand mode
    (config.training.compute_dtype)."""
    args = argparse.Namespace(batch=batch, iters=iters, steps=steps, warmup=warmup, config=config, dropout=dropout,
                              no_overlap=no_overlap, profile=profile, precision=precision)
    import torch.distributed as dist
    from configs import res64, res128
    from meshdiffusion_b200 import _native
    from meshdiffusion_b200.diffusion import sde_lib, trainer
    from meshdiffusion_b200.diffusion.evaler import load_grid_mask

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    own_group = world > 1 and not dist.is_initialized()
    if own_group:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    cfg = (res128 if args.config == "res128" else res64).get_config()
    if args.config == "tiny":  # test-size architecture (every layer type, seconds to build)
        cfg.data.image_size, cfg.model.nf, cfg.model.ch_mult = 16, 32, (1, 2)
        cfg.model.num_res_blocks, cfg.model.attn_resolutions = 1, (8,)
    cfg.model.compute_dtype = "bf16"
    cfg.training.compute_dtype = args.precision
    cfg.model.dropout = args.dropout
    cfg.training.iter_size = args.iters
    cfg.device = dev
    state = trainer.build_state(cfg, rank, world)
    model = state["model"]
    net = model.module
    R, B = cfg.data.image_size, args.batch
    mask = (load_grid_mask(R, dev) if R in (64, 128) else torch.ones(R, R, R, device=dev)).view(1, 1, R, R, R)
    net.mask.data[:] = mask
    # non-degenerate weights (the reference zero-inits Conv_1 / NIN_3 / head, which would make most gradients vanish)
    g = torch.Generator().manual_seed(7)
    with torch.no_grad():
        for n, p in net.named_parameters():
            if n.endswith("Conv_1.weight") or n.endswith("NIN_3.W") or (n.startswith("all_modules.") and p.dim() == 5 and p.shape[0] == 4):
                fan = p[0].numel() if p.dim() > 1 else 1
                p.copy_((torch.rand(p.shape, generator=g) * 2 - 1).to(p.device) * (3.0 / fan) ** 0.5)
    trainer.sync_replicas(state)
    sde = sde_lib.VPSDE(cfg.model.beta_min, cfg.model.beta_max, cfg.model.num_scales, device=dev)
    train_step_fn = trainer.make_train_step(cfg, state, sde, mask)
    if args.no_overlap:
        net.grad_overlap = False  # the product step with ONE blocking all-reduce inside optimize_fn, for comparison
    gen = torch.Generator(device=dev).manual_seed(42 + rank)
    data = [(torch.rand(B, 4, R, R, R, device=dev, generator=gen) * 2 - 1) * mask for _ in range(2)]

    # ---- device-time split: CUDA events around the product's own methods (they still run inside step_fn)
    ev = lambda: torch.cuda.Event(enable_timing=True)
    split = {"fwd": 0.0, "bwd": 0.0, "allreduce_exposed": 0.0, "weight_sync": 0.0}
    marks = []

    def timed(obj, name, key):
        fn = getattr(obj, name)

        def wrapper(*a, **k):
            e0, e1 = ev(), ev()
            e0.record()
            out = fn(*a, **k)
            e1.record()
            marks.append((key, e0, e1))
            return out
        setattr(obj, name, wrapper)

    timed(net, "_push_parameters", "weight_sync")
    orig_fwd = net._train_forward

    def fwd(x, labels):  # forward minus the parameter push it starts with
        e0, e1 = ev(), ev()
        e0.record()
        out = orig_fwd(x, labels)
        e1.record()
        marks.append(("fwd_incl_sync", e0, e1))
        return out
    net._train_forward = fwd
    timed(net, "_train_backward", "bwd")
    timed(net, "allreduce_grads", "allreduce_exposed")

    def one_step(step):
        last = None
        for it in range(args.iters):
            last = train_step_fn(state, data[(step + it) % 2], clear_grad=(it == 0), update_param=(it == args.iters - 1))["loss"]
        return last

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    losses = []
    for w in range(args.warmup):
        losses.append(one_step(w).item())
    barrier()
    marks.clear()
    t0, t1 = ev(), ev()
    t0.record()
    for s_ in range(args.steps):
        losses.append(one_step(args.warmup + s_))
    t1.record()
    barrier()
    losses = [float(v) for v in losses]
    ms = t0.elapsed_time(t1)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
    sync_ms = sum(a.elapsed_time(b) for k, a, b in marks if k == "weight_sync")
    split["weight_sync"] = sync_ms
    split["fwd"] = sum(a.elapsed_time(b) for k, a, b in marks if k == "fwd_incl_sync") - sync_ms
    split["bwd"] = sum(a.elapsed_time(b) for k, a, b in marks if k == "bwd")
    split["allreduce_exposed"] = sum(a.elapsed_time(b) for k, a, b in marks if k == "allreduce_exposed")
    split["other (loss, clip, Adam+EMA, host gaps)"] = ms - sum(split.values())
    L = _native.lib()
    fl, bf, nb, numel, arena = ctypes.c_double(), ctypes.c_double(), ctypes.c_int(), ctypes.c_longlong(), ctypes.c_longlong()
    _native.check(L.mdb_unet_info(net._train_handle, ctypes.byref(fl), ctypes.byref(arena), None, None))
    _native.check(L.mdb_unet_train_info(net._train_handle, ctypes.byref(bf), ctypes.byref(nb), ctypes.byref(numel)))
    samples = args.steps * args.iters * B * world
    peak = 1418.0
    try:
        peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["bf16_tflops_sustained"])
    except Exception:
        pass
    peak /= MMA_PER_PRODUCT[args.precision]  # algorithmic FLOPs: the split mode issues 3 MMAs per product
    tc_ms = split["fwd"] + split["bwd"]
    achieved = (fl.value + bf.value) * args.steps * args.iters * B / (tc_ms * 1e-3) / 1e12 if tc_ms > 0 else None
    if args.profile and rank == 0:
        x = data[0]
        lab = torch.full((B,), 500.0, device=dev)
        names = ctypes.create_string_buffer(1 << 18)
        msb = (ctypes.c_float * 4096)()
        n = ctypes.c_int()
        pred = orig_fwd(x, lab)
        _native.check(L.mdb_unet_profile_backward(net._train_handle, _native.ptr(pred), _native.ptr(net._flat_grad), B,
                                                  _native.current_stream(), names, len(names), msb, 4096, ctypes.byref(n)))
        rows = list(zip(names.value.decode().strip().split("\n"), [msb[i] for i in range(n.value)]))
        json.dump(rows, open(args.profile, "w"))
    result = None
    if rank == 0:
        result = ({
            "metric": f"training samples/s (res64 4x64^3 grids, {args.precision} operands, fp32 master/Adam/EMA)", "value": samples / (ms * 1e-3),
            "unit": "samples/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "dtype": args.precision, "data": "synthetic",
            "path": "product: trainer.make_train_step -> losses.get_step_fn -> FusedAdam(+EMA); all-reduce " +
                    ("blocking" if args.no_overlap else f"bucketed ({len(net._grad_buckets()) if world > 1 else 0} buckets) and overlapped with backward"),
            "config": {"workload": f"{args.config}.py train, micro-batch {B} x {args.iters} per GPU, dropout {args.dropout}, clip 1.0, Adam + EMA",
                       "global_batch": B * args.iters * world},
            "split_ms_per_step": {k: v / args.steps for k, v in split.items()},
            "flops_per_sample": {"forward": fl.value, "backward": bf.value},
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak if achieved else None,
                         "note": "forward + backward GEMM FLOPs / (fwd + bwd device time); peak = sustained bf16 / MMAs per product"},
            "bwd_launches": nb.value, "params": numel.value, "arena_bytes": arena.value, "losses": losses,
        })
    net.release_engine()
    if own_group:
        dist.destroy_process_group()
    return result


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=16, help="micro-batch per GPU")
    ap.add_argument("--iters", type=int, default=4, help="micro-batches per optimiser step (batch*iters = 64/GPU in BASELINE)")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--config", default="res64", choices=["res64", "res128", "tiny"])
    ap.add_argument("--dropout", type=float, default=0.1)
    ap.add_argument("--no-overlap", action="store_true", help="one blocking all-reduce after the backward pass instead of buckets")
    ap.add_argument("--profile", default=None, help="write per-launch device times of one forward+backward as JSON")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "bf16x3"], help="training operand mode (config.training.compute_dtype)")
    a = ap.parse_args()
    out = run(a.batch, a.iters, a.steps, a.warmup, a.config, a.dropout, a.no_overlap, a.profile, a.precision)
    if out is not None:
        print(json.dumps(out))


if __name__ == "__main__":
    main()

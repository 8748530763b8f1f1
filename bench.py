#!/usr/bin/env python
"""Benchmark of the hot path: denoising steps of the res64 unconditional sampler (BASELINE.json configs[1]).

    python bench.py --gpus N --steps K --warmup W            # this repo, N ranks (torchrun for N > 1)
    python bench.py --impl reference --steps K --warmup W    # the unmodified reference modules on the host cores
    python bench.py --res 128 --strong --gpus N              # BASELINE configs[3]: 8 grids in total, 8/N per GPU
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR   # also write the outputs of the last timed step

A "step" is one denoising step of pc_sampler for one batch: U-Net evaluation + ancestral update over
[batch, 4, 64, 64, 64]. metric = sample-steps/s = batch * steps / time, whole job (sum over ranks).

The HEADLINE is measured in the operand mode that meets north_star's parity contract (1e-3 against the reference's
fp32 arithmetic): `bf16x3`, split-bf16 operands (hi*hi + hi*lo + lo*hi into the fp32 TMEM accumulator). The same line
carries complete secondary legs (`legs`: value, e2e, roofline, clocks each) for `tf32` operands (the arithmetic class of
the reference's own stock GPU path, 1.3e-3) and plain `bf16` operands (throughput mode, 1.2e-2).

  value     : device-resident loop (mdb_sampler_run: state, noise and coefficients never leave HBM), CUDA events.
  e2e       : same steps through the public Python API (model(x, labels) + fused update) with the state copied
              host->device from pinned memory before and device->host after EVERY step.
  roofline  : the tcgen05 implicit-GEMM kernel: algorithmic FLOPs / CUDA-event time of exactly those launches inside
              one forward, against the measured sustained bf16 cuBLAS peak (MEASURED_PEAKS.json) divided by the tensor
              instructions the mode issues per product (1 bf16, 2 tf32, 3 bf16x3).
  cpu_baseline       : the unmodified reference modules (baseline/_ref) on the host cores, B=1 (bounded sample).
  torch_gpu_baseline : the same reference modules under stock PyTorch on the same B200 (TF32 default / strict fp32 /
                       bf16 autocast) -- the same-box stand-in for the "1x A100-equivalent PyTorch-GPU" figure.
  train     : BASELINE configs[2], one optimiser step of the PRODUCT training path (tools/bench_train.py), all ranks.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "denoising sample-steps/sec at res-64 (4x64^3), uncond_gen PC sampler"
UNIT = "sample-steps/s"
N_EVALS_FULL = 999  # pc_sampler's unconditional loop evaluates the network N-1 = 999 times (sampling.py:471)
MMA_PER_PRODUCT = {"bf16": 1.0, "tf32": 2.0, "bf16x3": 3.0}
PARITY = {"bf16x3": "fp32-class: full res64 net 4e-5 max-rel vs the fp32 oracle, gate 1e-3 = north_star's tolerance (tests/test_gpu_unet.py)",
          "tf32": "1.6e-3 vs fp32 on the full res64 net (the reference's own stock TF32 GPU path: 1.3e-3), gate 3e-3",
          "bf16": "1.3e-2 vs fp32 on the full res64 net (throughput mode), gate 4e-2"}


def host_threads():
    """oneDNN conv3d scales to ~32 threads on this host class and gets slower beyond (measured on the 128-core GPU box:
    16 thr 6.7 s, 32 thr 6.1 s, 64 thr 8.3 s, 128 thr 46 s per res64 forward) -- use what is actually useful."""
    return int(os.environ.get("MDB_CPU_THREADS", min(32, os.cpu_count() or 1)))


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clock / throttle sampling during the timed region."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        rows = [r for r in self.rows if len(r) >= 7]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        sm = sorted(float(r[0]) for r in rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][1]), "reasons": reasons,
                "power_w_max": max(float(r[2]) for r in rows), "samples": len(rows)}


def build_model(precision, batch, device, res=64):
    from configs import res64, res128
    from meshdiffusion_b200.diffusion.models import utils as mutils
    from meshdiffusion_b200.diffusion.models.init_utils import random_init_nondegenerate
    cfg = (res128 if res == 128 else res64).get_config()
    cfg.model.compute_dtype = precision
    cfg.model.engine_max_batch = batch
    cfg.device = device
    torch.manual_seed(0)
    model = mutils.create_model(cfg)
    random_init_nondegenerate(model.module)
    model.eval()
    return cfg, model


class Ctx:
    """Process-group plumbing shared by the legs."""

    def __init__(self):
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.device = torch.device(f"cuda:{self.local}")
        self.dist = None
        if self.world > 1:
            os.environ.setdefault("NCCL_DEBUG", "WARN")  # keep stdout to the single JSON line
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=self.device)
            self.dist = dist

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, ms):
        if self.dist is None:
            return ms
        t = torch.tensor([ms], device=self.device)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.item()


def sampler_leg(ctx, precision, B, R, K, W, dump_profile=None, full_run=False, dump_outputs=False):
    """One operand mode: device-resident loop, end-to-end loop, roofline of the GEMM launches, clocks. With `dump_outputs`
    the leg also returns what the last timed step of the device-resident loop left for its caller (the state x and
    x_mean), sampled by `output_sample`."""
    from meshdiffusion_b200.diffusion import sde_lib, sampling
    from meshdiffusion_b200.geometry.dmtet import grid_mask_from_tets
    device, world, rank = ctx.device, ctx.world, ctx.rank
    cfg, model = build_model(precision, B, device, R)
    net = model.module
    sde = sde_lib.VPSDE(cfg.model.beta_min, cfg.model.beta_max, cfg.model.num_scales, device=device)
    mask = grid_mask_from_tets(R).to(device)
    net.mask.data[:] = mask.view(1, 1, R, R, R)
    mask_flat = mask.reshape(-1).contiguous()
    timesteps = torch.linspace(sde.T, 1e-3, sde.N, device=device)
    idx = (timesteps * (sde.N - 1)).long()
    # a window of more than N steps runs on into the schedule again from its first step, so --warmup + --steps can be
    # any length
    cyclic = lambda v: [v[i % len(v)] for i in range(max(len(v), W + K))]
    labels_all = cyclic((timesteps * (sde.N - 1)).cpu().tolist())
    betas = cyclic(sde.discrete_betas[idx].cpu().tolist())
    stds = cyclic(sde.sqrt_1m_alphas_cumprod[idx].cpu().tolist())
    g = torch.Generator(device=device).manual_seed(42 + rank)
    x = (torch.randn(B, 4, R, R, R, device=device, generator=g) * mask).contiguous()

    def native_steps(first, n):
        return sampling._native_loop(net, x, mask_flat, labels_all, betas, stds, n, 42 + rank, first)

    # ---- device-resident loop ("value")
    native_steps(0, W)
    ctx.barrier()
    clocks = ClockSampler(ctx.local)
    clocks.start()
    try:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        x_mean = native_steps(W, K)
        e1.record()
        ctx.barrier()
    finally:
        clk = clocks.stop()
    ms = ctx.max_over_ranks(e0.elapsed_time(e1))
    value = world * B * K / (ms * 1e-3)
    outputs = {f"{precision}_x": output_sample(x), f"{precision}_x_mean": output_sample(x_mean)} if dump_outputs else None

    # ---- the complete 999-evaluation run (opt-in: minutes), so samples/s is measured rather than extrapolated
    full = None
    if full_run:
        x.copy_(torch.randn(B, 4, R, R, R, device=device, generator=g) * mask)
        ctx.barrier()
        e0.record()
        out = native_steps(0, N_EVALS_FULL)
        e1.record()
        ctx.barrier()
        ms_full = ctx.max_over_ranks(e0.elapsed_time(e1))
        full = {"samples_per_s": world * B / (ms_full * 1e-3), "seconds": ms_full * 1e-3, "evals": N_EVALS_FULL,
                "finite": bool(torch.isfinite(out).all())}

    # ---- end to end through the public API with host buffers every step ("e2e")
    host_x = torch.empty(B, 4, R, R, R, pin_memory=True)
    host_x.copy_(x.cpu())
    host_out = torch.empty(B, 4, R, R, R, pin_memory=True)
    vec = torch.ones(B, device=device)

    def api_step(i):
        xd = host_x.to(device, non_blocking=True)
        eps = model(xd, vec * labels_all[i])
        xd, x_mean = sampling._fused_update(eps, xd, torch.randn_like(xd), mask_flat, betas[i], stds[i])
        host_out.copy_(x_mean, non_blocking=True)
        host_x.copy_(xd, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    with net.frozen():  # what pc_sampler does around its loop: weights cannot change between steps
        for i in range(W):
            api_step(i)
        ctx.barrier()
        e0.record()
        for i in range(W, W + K):
            api_step(i)
        e1.record()
        ctx.barrier()
    ms_e2e = ctx.max_over_ranks(e0.elapsed_time(e1))
    state_bytes = B * 4 * R ** 3 * 4

    # ---- roofline of the dominant kernel (rank 0): per-launch CUDA events inside one forward
    roofline, launches_per_forward, info = None, None, net.engine_info()
    if rank == 0:
        labels = vec * labels_all[W]
        prof = net.profile(x, labels)
        if dump_profile:
            with open(dump_profile, "w") as f:
                json.dump(prof, f)
        launches_per_forward = len(prof) + 2  # + stats memset, + second kernel of the temb step
        conv_ms = sum(t for n, t in prof if _is_conv_gemm(n))
        all_gemm_ms = sum(t for n, t in prof if _is_gemm(n))
        peaks, src = measured_peaks()
        flops = info["flops_per_sample"] * B
        # FLOPs of the non-conv GEMMs (attention, stem) are < 3 % of the total; the roofline is quoted on all launches of
        # the tcgen05 kernel together: algorithmic FLOPs / their summed duration
        per = MMA_PER_PRODUCT[precision]
        peak = peaks["bf16_tflops_sustained"] / per
        ach = flops / (all_gemm_ms * 1e-3) / 1e12
        fwd_ms = sum(t for _, t in prof)
        roofline = {"bound": "tensor", "kernel": "gemm_tc_kernel (tcgen05 implicit-GEMM conv3d / NIN / attention)",
                    "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "traffic": ncu_traffic(precision),
                    "peak_source": f"{src} bf16_tflops_sustained" + (f" / {per:g} ({precision}: {per:g} bf16-rate tensor instructions per product)" if per != 1 else ""),
                    "issued_tflops": ach * per, "gemm_ms_per_forward": all_gemm_ms, "conv_ms_per_forward": conv_ms,
                    "forward_ms": fwd_ms, "non_gemm_share_of_forward": 1.0 - all_gemm_ms / fwd_ms,
                    "gemm_launches_per_forward": info["gemm_launches"],
                    "algorithmic_flops_per_launch_avg": flops / info["gemm_launches"]}
    leg = {"dtype": precision, "parity": PARITY[precision], "value": value, "unit": UNIT, "ms_per_step": ms / K,
           "samples_per_s_extrapolated": value / N_EVALS_FULL, "full_run": full,
           "e2e": {"value": world * B * K / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": state_bytes,
                   "d2h_bytes_per_step": 2 * state_bytes, "ms_per_step": ms_e2e / K},
           "gpu_launches": int(K * (launches_per_forward + 2)) if launches_per_forward else None,
           "clocks": clk, "roofline": roofline, "engine": info}
    net.release_engine()
    del model, net
    torch.cuda.empty_cache()
    return leg, mask, outputs


def output_sample(t, n=1 << 21):
    """float32 copy of at most `n` elements of `t`: all of them, or a fixed seeded sample (sorted flat indices, the same for
    every run and build) of a larger tensor. 2^21 elements keep the six arrays of three operand modes at 48 MB."""
    flat = t.detach().reshape(-1)
    if flat.numel() > n:
        idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(0))[:n].sort().values
        flat = flat[idx.to(flat.device)]
    return flat.float().cpu().numpy()


def ncu_traffic(precision):
    """dram read+write bytes per launch of the dominant launch type (128->128 conv @64^3) from the committed `ncu --set full`
    capture of this mode (taken at batch 8; reported as captured, with its batch and source file), or null."""
    name = {"bf16": "r02_ncu_conv_final_bf16.txt", "bf16x3": "r02_ncu_conv_final_bf16x3.txt", "tf32": "r02_ncu_conv_final_tf32.txt"}[precision]
    path = os.path.join(ROOT, "profiles", name)
    try:
        rd = wr = None
        for line in open(path):
            if "dram__bytes_read.sum =" in line and rd is None:
                v, u = line.split("=")[1].split()[:2]; rd = float(v) * (1e9 if u.startswith("G") else 1e6)
            if "dram__bytes_write.sum =" in line and wr is None:
                v, u = line.split("=")[1].split()[:2]; wr = float(v) * (1e9 if u.startswith("G") else 1e6)
        es = 2 if precision == "bf16" else 4
        return {"bytes_per_launch": rd + wr, "batch": 8, "launch": "conv3x3x3 128->128 @64^3", "source": f"profiles/{name} (static capture, not this run)",
                "algorithmic_bytes_per_launch": 2 * 8 * 64 ** 3 * 128 * es + 27 * 128 * 128 * es * (1.5 if precision == "bf16x3" else 1)}
    except Exception:
        return None


def _is_gemm(name):
    return (".conv" in name or ".nin" in name or name.endswith(".gemm") or name.endswith(".qk") or name.endswith(".pv")
            or name.endswith(".proj") or name.startswith("down"))


def _is_conv_gemm(name):
    return ".conv" in name or name.startswith("down")


def cpu_baseline(steps=1):
    """The unmodified reference modules on the host cores: B=1, `steps` steps of pc_sampler after one warm-up."""
    from baseline import reference_arm
    threads = host_threads()
    torch.set_num_threads(threads)
    if not reference_arm.available():
        return {"error": "baseline/_ref missing (python baseline/install_reference.py)"}
    ref, config, model, sde, mask = reference_arm.build("cpu")
    reference_arm.run_steps(ref, config, model, sde, mask, 1, 1)
    dt = reference_arm.run_steps(ref, config, model, sde, mask, 1, steps)
    return {"value": steps / dt, "unit": UNIT, "cores": threads, "kind": "reference",
            "sample": f"B=1, {steps} step(s) of the same res64 sampler after 1 warm-up: unmodified reference modules (baseline/_ref) through "
                      "get_sampling_fn -> pc_sampler, torch CPU fp32", "s_per_step": dt / steps}


def run_ours(args):
    ctx = Ctx()
    B, R, K, W = args.batch, args.res, args.steps, args.warmup
    if args.strong:
        if B % ctx.world != 0:
            raise SystemExit(f"--strong: {B} grids do not divide over {ctx.world} ranks")
        B //= ctx.world
    precisions = [args.precision] + [p for p in args.legs.split(",") if p and p != args.precision]
    legs, mask, outputs = {}, None, {}
    for i, prec in enumerate(precisions):
        legs[prec], mask, out = sampler_leg(ctx, prec, B, R, K, W, dump_profile=args.dump_profile if i == 0 else None,
                                            full_run=args.full_run and i == 0, dump_outputs=bool(args.dump_outputs) and ctx.rank == 0)
        if out:
            outputs.update(out)
        if ctx.rank == 0:  # progress on stderr (stdout carries only the final JSON line)
            print(f"[bench] {prec}: value {legs[prec]['value']:.2f} e2e {legs[prec]['e2e']['value']:.2f} {UNIT}, "
                  f"gemm frac {legs[prec]['roofline']['frac']:.3f}", file=sys.stderr, flush=True)
    head = legs[args.precision]

    cpu = torch_gpu = None
    if ctx.rank == 0 and ctx.world == 1 and R == 64:
        if not args.no_cpu_baseline:
            try:
                cpu = cpu_baseline(steps=1)
            except Exception as ex:  # a reported baseline: never fails the bench line
                cpu = {"error": str(ex)[:200]}
        if not args.no_torch_gpu_baseline:
            try:
                from baseline import reference_arm
                torch_gpu = reference_arm.gpu_baseline(batch=8, steps=3, warmup=1, device=f"cuda:{ctx.local}") if reference_arm.available() else {"error": "baseline/_ref missing"}
            except Exception as ex:
                torch_gpu = {"error": str(ex)[:200]}
            torch.cuda.empty_cache()

    # ---- BASELINE configs[2]: one optimiser step of the product training path, on every rank (data-parallel for N > 1)
    train = None
    if not args.no_train_leg and R == 64:
        torch.cuda.empty_cache()
        try:
            sys.path.insert(0, os.path.join(ROOT, "tools"))
            import bench_train
            t = bench_train.run(batch=16, iters=1, steps=2, warmup=1, config="res64", dropout=0.1, no_overlap=False, profile=None)
            if ctx.rank == 0:
                train = {"value": t["value"], "unit": t["unit"], "n_gpus": t["n_gpus"], "path": t["path"], "workload": t["config"]["workload"],
                         "ms_per_step": t["ms_per_step"], "split_ms_per_step": t["split_ms_per_step"],
                         "fwd_bwd_tflops": t["roofline"]["achieved"], "fwd_bwd_frac_of_peak": t["roofline"]["frac"]}
        except Exception as ex:  # informational leg: never fails the bench line
            train = {"error": str(ex)[:300]}

    if ctx.rank == 0:
        line = {
            "metric": METRIC if R == 64 else METRIC.replace("res-64 (4x64^3)", "res-128 (4x128^3)"), "value": head["value"], "unit": UNIT,
            "n_gpus": ctx.world, "steps": K, "warmup": W, "ms_per_step": head["ms_per_step"], "higher_is_better": True,
            "scaling": "strong" if args.strong else "weak", "vs_baseline": None,
            "dtype": args.precision, "data": "synthetic (random-init non-degenerate weights, N(0,1)*grid_mask state)",
            "config": {"workload": f"res{R}.py uncond_gen, batch={B}/GPU" + (f" ({B * ctx.world} in total, strong scaling)" if args.strong else "") +
                                   ", PC sampler (ancestral_sampling + none), steps of the N=1000 schedule",
                       "batch_per_gpu": B, "image_size": R, "precision": args.precision, "parity": head["parity"],
                       "l2_policy": "inputs larger than L2: per-step activation working set is several GB at batch 32"},
            "samples_per_s": head["full_run"]["samples_per_s"] if head["full_run"] else head["samples_per_s_extrapolated"],
            "samples_per_s_is": "measured over the full 999-evaluation run" if head["full_run"] else "extrapolated: value / 999 (pass --full-run to measure it)",
            "e2e": head["e2e"], "gpu_launches": head["gpu_launches"], "clocks": head["clocks"], "roofline": head["roofline"],
            "cpu_baseline": cpu, "torch_gpu_baseline": torch_gpu,
            "legs": {p: legs[p] for p in precisions if p != args.precision},
            "engine": head["engine"], "full_run": head["full_run"], "train": train,
        }
        print(json.dumps(line))
    if outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in outputs.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    if ctx.dist is not None:
        ctx.dist.destroy_process_group()


def run_reference(args):
    """Reference arm: the UNMODIFIED reference modules from baseline/_ref through the reference's own public API
    (mutils.create_model, sampling.get_sampling_fn -> pc_sampler) on the host cores; this repository's package is not
    imported. Each step = a bounded sample of the workload: 1 of the 32 grids of the batch."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from baseline import reference_arm
    K, W = args.steps, args.warmup
    if not reference_arm.available():
        print(json.dumps({"impl": "reference", "unavailable": "baseline/_ref is missing (built by __graft_entry__.build() where /root/reference exists)"}))
        return
    threads = host_threads()
    torch.set_num_threads(threads)
    ref, config, model, sde, mask = reference_arm.build("cpu")
    if W > 0:
        reference_arm.run_steps(ref, config, model, sde, mask, 1, W)
    dt = reference_arm.run_steps(ref, config, model, sde, mask, 1, K)
    value = K / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": K, "warmup": W,
        "ms_per_step": dt / K * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": "res64.py uncond_gen PC sampler; each step = a bounded sample (1 of the 32 grids of the batch) on the host cores",
                   "batch_per_step": 1, "image_size": 64},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "reference",
                         "sample": "1 grid of the 32-grid batch per step (U-Net evaluation + ancestral update): unmodified reference modules "
                                   "(baseline/_ref), get_sampling_fn -> pc_sampler, torch CPU fp32"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=None, help="grids per GPU (default 32 = BASELINE configs[1]; 8 with --res 128 = configs[3]); with --strong: grids in total")
    ap.add_argument("--res", type=int, default=64, choices=[64, 128], help="64 = the metric's config (default); 128 = BASELINE configs[3] (secondary)")
    ap.add_argument("--strong", action="store_true", help="strong scaling: --batch grids in total, split over the ranks (BASELINE configs[3]: 8 -> 8/4/2/1 per GPU)")
    ap.add_argument("--precision", default="bf16x3", choices=["bf16x3", "tf32", "bf16"], help="operand mode of the headline (default: the parity-grade mode)")
    ap.add_argument("--legs", default=None, help="comma-separated secondary operand modes measured in full (default: tf32,bf16 at res 64, none at res 128)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--full-run", action="store_true", help="also run the complete 999-evaluation loop (minutes) so samples/s is measured")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-torch-gpu-baseline", action="store_true")
    ap.add_argument("--no-train-leg", action="store_true", help="skip the training-step measurement (tools/bench_train.py)")
    ap.add_argument("--dump-profile", default=None, help="write the per-launch CUDA-event times of one forward as JSON")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write what the last timed step of each operand mode's device-resident loop returned (rank 0: state x "
                         "and x_mean) as DIR/<mode>_x.npy and DIR/<mode>_x_mean.npy, float32, a fixed seeded sample of at "
                         "most 2^21 elements each; the inputs depend only on the arguments, so two builds compare output for output")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.batch is None:
        args.batch = 8 if args.res == 128 else 32
    if args.legs is None:
        args.legs = "tf32,bf16" if args.res == 64 else ""
    if args.impl == "reference":
        run_reference(args)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: the hot path has no CPU fallback (use --impl reference for the CPU arm)")
    run_ours(args)


if __name__ == "__main__":
    main()

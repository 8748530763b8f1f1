"""Score networks `ddpm_res64` / `ddpm_res128` backed by the sm_100a engine.

Drop-in for the reference's DDPMRes64 / DDPMRes128 (lib/diffusion/models/ddpm_res64.py:39-199,
ddpm_res128.py:41-215): same registered names, same `model(x, labels)` call, same parameter names and shapes
(so reference checkpoints load with `load_state_dict`), same `.mask` / `.coords` / `sigmas` entries. The module
holds the fp32 master parameters as ordinary torch Parameters; the forward pass runs entirely inside
libmeshdiff_b200.so (tcgen05 implicit-GEMM convolutions + fused bandwidth kernels). There is no PyTorch or CPU
fallback: calling the model without the native library and a CUDA device raises.
"""
import ctypes
import math

import numpy as np
import torch
import torch.nn as nn

from ... import _native
from . import utils


PRECISIONS = {"bf16": 0, "tf32": 1, "bf16x3": 2}  # include/meshdiff_b200.h: mdb_unet_config.precision
TRAIN_PRECISIONS = ("bf16", "bf16x3")  # the engine builds no tf32 training plan


def arch_from_config(config):
    """Structural hyper-parameters read by the reference constructors (ddpm_res64.py:46-53, ddpm_res128.py:48-55)."""
    is128 = config.model.name.startswith("ddpm_res128")
    return dict(
        image_size=int(config.data.image_size), nf=int(config.model.nf),
        ch_mult=tuple(int(c) for c in config.model.ch_mult), num_res_blocks=int(config.model.num_res_blocks),
        attn_resolutions=tuple(int(r) for r in config.model.attn_resolutions),
        num_channels=int(config.data.num_channels), stem_ksize=5 if is128 else 3, use_pos_bias=not is128,
        level0_blocks=2 if is128 else int(config.model.num_res_blocks),
    )


def _config_c(arch, max_batch, precision, training=False):
    c = _native.UNetConfigC()
    c.image_size, c.nf, c.n_levels = arch["image_size"], arch["nf"], len(arch["ch_mult"])
    for i, v in enumerate(arch["ch_mult"]):
        c.ch_mult[i] = v
    c.num_res_blocks, c.level0_blocks = arch["num_res_blocks"], arch["level0_blocks"]
    c.n_attn = len(arch["attn_resolutions"])
    for i, v in enumerate(arch["attn_resolutions"]):
        c.attn_resolutions[i] = v
    c.num_channels, c.stem_ksize = arch["num_channels"], arch["stem_ksize"]
    c.use_pos_bias = 1 if arch["use_pos_bias"] else 0
    c.max_batch, c.precision = max_batch, PRECISIONS[precision]
    c.training = 1 if training else 0
    return c


def param_table(arch):
    """[(name, shape)] in engine order, from a GPU-less dry plan of the native library."""
    L = _native.lib()
    h = ctypes.c_void_p()
    cfg = _config_c(arch, 1, "bf16")
    _native.check(L.mdb_unet_create_dry(ctypes.byref(cfg), ctypes.byref(h)))
    try:
        out = []
        for i in range(L.mdb_unet_num_params(h)):
            name, numel, nd = ctypes.c_char_p(), ctypes.c_longlong(), ctypes.c_int()
            shape = (ctypes.c_longlong * 8)()
            _native.check(L.mdb_unet_param_info(h, i, ctypes.byref(name), ctypes.byref(numel), ctypes.byref(nd), shape))
            out.append((name.value.decode(), tuple(int(shape[j]) for j in range(nd.value))))
        return out
    finally:
        L.mdb_unet_destroy(h)


def variance_scaling_uniform(shape, scale=1.0, generator=None):
    """`default_init(scale)` of the reference (layers.py:54-91): fan_avg, uniform, in_axis=1 / out_axis=0."""
    scale = 1e-10 if scale == 0 else scale
    receptive = 1
    for d in shape[2:]:
        receptive *= d
    fan_in, fan_out = shape[1] * receptive, shape[0] * receptive
    bound = math.sqrt(3.0 * scale / ((fan_in + fan_out) / 2.0))
    return (torch.rand(shape, generator=generator) * 2.0 - 1.0) * bound


def make_grad_buckets(entries, total_numel, bucket_bytes):
    """entries: (offset, numel, ready_launches) of every slot of the flat gradient buffer. Returns [(ready, lo, hi)] sorted
    by readiness: contiguous, disjoint ranges that tile [0, total_numel), cut from the END of the buffer (the head's
    gradients are final first, the time-embedding MLP's last) in pieces of at least `bucket_bytes`; a range is ready once
    every gradient inside it is final."""
    buckets, hi, ready = [], total_numel, 0
    for off, numel, rdy in sorted(entries, reverse=True):
        ready = max(ready, rdy)
        if (hi - off) * 4 >= bucket_bytes:
            buckets.append((ready, off, hi))
            hi, ready = off, 0
    if hi > 0:
        buckets.append((ready, 0, hi))
    buckets.sort()
    return buckets


class _ScoreNetFn(torch.autograd.Function):
    """Autograd node of the whole score network: forward and backward both run inside the native engine, so the stock
    `loss.backward()` of the reference's step_fn (losses.py:104-139) works unchanged. Parameter gradients are written
    by the engine straight into the module's flat fp32 gradient buffer (`p.grad` are views of it)."""

    @staticmethod
    def forward(ctx, net, x, labels, *params):
        out = net._train_forward(x, labels)
        ctx.net = net
        ctx.save_for_backward(x, labels)
        return out

    @staticmethod
    def backward(ctx, dout):
        x, labels = ctx.saved_tensors
        ctx.net._train_backward(x, labels, dout)
        return (None, None, None) + (None,) * len(ctx.net._trainable)


class _Scope(nn.Module):
    """Plain container so dotted parameter names become nested state-dict keys."""


class ScoreNet(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.arch = arch_from_config(config)
        # inference operand mode; the default is the parity-grade one (results within 1e-3 of the reference's fp32 arithmetic).
        # 'tf32' (1.6e-3, 1.55x faster) and 'bf16' (1.3e-2, 2.7x faster) are opt-in.
        self.precision = str(config.model.get("compute_dtype", "bf16x3")) if hasattr(config.model, "get") else "bf16x3"
        if self.precision not in PRECISIONS:
            raise ValueError("config.model.compute_dtype must be 'bf16', 'tf32' or 'bf16x3'")
        # training operand mode: 'bf16' (the default) or 'bf16x3' (split bf16 forward, data and weight gradients:
        # fp32-class gradients at about a third of the bf16 tensor rate)
        training = getattr(config, "training", None)
        self.train_precision = str(training.get("compute_dtype", "bf16")) if hasattr(training, "get") else "bf16"
        if self.train_precision not in TRAIN_PRECISIONS:
            raise ValueError("config.training.compute_dtype must be 'bf16' or 'bf16x3'")
        self.max_batch = int(config.model.get("engine_max_batch", 0) or 0) if hasattr(config.model, "get") else 0
        self.scale_by_sigma = bool(config.model.scale_by_sigma)
        self.dropout = float(config.model.get("dropout", 0.0)) if hasattr(config.model, "get") else 0.0
        self._train_handle, self._train_batch, self._train_synced = None, 0, None
        self._flat_grad, self._drop_calls, self._pending = None, 0, None
        # data-parallel training: when True (the trainer sets it for the last micro-batch of an optimiser step) the backward
        # pass all-reduces finished gradient buckets on a side stream while the remaining launches run
        self.reduce_in_backward = False
        self.grad_overlap = bool(config.model.get("grad_overlap", True)) if hasattr(config.model, "get") else True
        self.bucket_bytes = int(config.model.get("grad_bucket_mb", 64)) << 20 if hasattr(config.model, "get") else 64 << 20
        self._buckets, self._pending_reduce, self._side_stream = None, None, None
        # same buffer as the reference (ddpm_res64.py:44): float64 [num_scales]
        self.register_buffer("sigmas", torch.tensor(utils.get_sigmas(config)))
        self._names = []
        head_idx = None
        table = param_table(self.arch)
        for name, _ in table:
            if name.startswith("all_modules."):
                head_idx = max(head_idx or 0, int(name.split(".")[1]))
        # registration order == the reference's parameters() order (own Parameters, pos_layer, mask_layer,
        # all_modules.*), because the EMA checkpoint stores a positional list (ema.py:91-98)
        def ref_order(item):
            n = item[0]
            if n == "coords": return (0, 0)
            if n == "mask": return (1, 0)
            if n.startswith("pos_layer."): return (2, 0)
            if n.startswith("mask_layer."): return (3, 0)
            return (4, int(n.split(".")[1]))
        for name, shape in sorted(table, key=ref_order):
            self._register(name, self._initial_value(name, shape, head_idx), trainable=name not in ("mask", "coords"))
        self._handle = None
        self._engine_batch = 0
        self._synced = None
        self._trainable = [n for n in self._names if n not in ("mask", "coords")]

    # ---- parameter plumbing -------------------------------------------------------------------------------------
    def _initial_value(self, name, shape, head_idx):
        leaf = name.split(".")[-1]
        if name == "mask" or name == "coords":
            return torch.zeros(shape)
        if leaf in ("bias", "b"):
            return torch.zeros(shape)
        if "GroupNorm" in name or name == f"all_modules.{head_idx - 1}.weight":
            return torch.ones(shape)
        if leaf == "W":  # NIN: init_scale 0.1, except NIN_3 (0.) -- layers.py:574-576,593
            return variance_scaling_uniform(shape, 0.0 if name.endswith("NIN_3.W") else 0.1)
        zero_init = name.endswith("Conv_1.weight") or name == f"all_modules.{head_idx}.weight"
        return variance_scaling_uniform(shape, 0.0 if zero_init else 1.0)

    def _register(self, dotted, value, trainable):
        parts = dotted.split(".")
        node = self
        for p in parts[:-1]:
            if not hasattr(node, p):
                node.add_module(p, _Scope())
            node = getattr(node, p)
        node.register_parameter(parts[-1], nn.Parameter(value, requires_grad=trainable))
        self._names.append(dotted)

    def _param(self, dotted):
        node = self
        for p in dotted.split("."):
            node = getattr(node, p)
        return node

    # ---- engine --------------------------------------------------------------------------------------------------
    def _ensure_engine(self, batch, device):
        L = _native.lib()
        if self._handle is not None and batch <= self._engine_batch:
            return
        if device.type != "cuda":
            raise _native.NativeError("the score network runs only on a CUDA (sm_100a) device; there is no CPU path")
        self.release_engine()
        mb = max(batch, self.max_batch)
        cfg = _config_c(self.arch, mb, self.precision)
        h = ctypes.c_void_p()
        with torch.cuda.device(device):
            _native.check(L.mdb_unet_create(ctypes.byref(cfg), ctypes.byref(h)))
        self._handle, self._engine_batch, self._synced = h, mb, None

    def release_engine(self):
        if self._handle is not None:
            _native.lib().mdb_unet_destroy(self._handle)
            self._handle = None
        if getattr(self, "_train_handle", None) is not None:
            _native.lib().mdb_unet_destroy(self._train_handle)
            self._train_handle = None

    # ---- training engine (bf16 or split-bf16 operands, fp32 master parameters and gradients) ----------------------
    def _ensure_train_engine(self, batch, device):
        L = _native.lib()
        if self._train_handle is not None and batch <= self._train_batch:
            return
        if device.type != "cuda":
            raise _native.NativeError("the score network trains only on a CUDA (sm_100a) device; there is no CPU path")
        if self._train_handle is not None:
            L.mdb_unet_destroy(self._train_handle)
            self._train_handle = None
        cfg = _config_c(self.arch, batch, self.train_precision, training=True)
        h = ctypes.c_void_p()
        with torch.cuda.device(device):
            _native.check(L.mdb_unet_create(ctypes.byref(cfg), ctypes.byref(h)))
        self._train_handle, self._train_batch, self._train_synced = h, batch, None
        numel = ctypes.c_longlong()
        _native.check(L.mdb_unet_train_info(h, None, None, ctypes.byref(numel)))
        if self._flat_grad is None or self._flat_grad.numel() != numel.value or self._flat_grad.device != device:
            self._flat_grad = torch.zeros(numel.value, dtype=torch.float32, device=device)
            self._grad_views = {}
            for n in self._trainable:
                off = ctypes.c_longlong()
                _native.check(L.mdb_unet_grad_offset(h, n.encode(), ctypes.byref(off)))
                p = self._param(n)
                self._grad_views[n] = self._flat_grad[off.value:off.value + p.numel()].view(p.shape)
        self._buckets = None

    def _grad_buckets(self):
        """[(ready_launches, lo, hi)] covering the flat gradient buffer from its END (the head's gradients are final first,
        the time-embedding MLP's last) in pieces of ~bucket_bytes; a bucket is ready when every gradient in it is final."""
        if self._buckets is not None:
            return self._buckets
        L = _native.lib()
        entries = []
        for n in self._names:
            off, rdy = ctypes.c_longlong(), ctypes.c_int()
            _native.check(L.mdb_unet_grad_offset(self._train_handle, n.encode(), ctypes.byref(off)))
            _native.check(L.mdb_unet_grad_ready(self._train_handle, n.encode(), ctypes.byref(rdy)))
            entries.append((off.value, self._param(n).numel(), rdy.value))
        self._buckets = make_grad_buckets(entries, self._flat_grad.numel(), self.bucket_bytes)
        return self._buckets

    def _backward_with_overlapped_allreduce(self, dout, B, accumulate):
        """mdb_unet_backward_marked + one NCCL all-reduce (mean) per bucket on a side stream, each starting as soon as the
        launches that write its gradients have retired. The optimiser's allreduce_grads() call then only waits."""
        import torch.distributed as dist
        L = _native.lib()
        buckets = self._grad_buckets()
        if self._side_stream is None:
            self._side_stream = torch.cuda.Stream(device=self._flat_grad.device)
            self._events = [torch.cuda.Event() for _ in buckets]
            for e in self._events:
                e.record()  # materialises the cudaEvent_t handles
        n = len(buckets)
        steps = (ctypes.c_int * n)(*[b[0] for b in buckets])
        handles = (ctypes.c_void_p * n)(*[e.cuda_event for e in self._events])
        _native.check(L.mdb_unet_backward_marked(self._train_handle, _native.ptr(dout), _native.ptr(self._flat_grad), self._flat_grad.numel(),
                                                 B, 1 if accumulate else 0, steps, handles, n, _native.current_stream()))
        works = []
        with torch.cuda.stream(self._side_stream):
            for (rdy, lo, hi), ev in zip(buckets, self._events):
                self._side_stream.wait_event(ev)
                works.append(dist.all_reduce(self._flat_grad[lo:hi], op=dist.ReduceOp.AVG, async_op=True))
        self._pending_reduce = works

    def _push_parameters(self, handle, synced):
        """set_param for every tensor whose fingerprint differs from `synced`, then commit. Returns the fingerprints."""
        L = _native.lib()
        fp = self._fingerprints()
        changed = None if synced is None else (fp != synced).nonzero().flatten().tolist()
        if changed is not None and not changed:
            return fp
        stream = _native.current_stream()
        self._upload(handle, range(len(self._names)) if changed is None else changed, stream)
        torch.cuda.current_stream().synchronize()
        _native.check(L.mdb_unet_commit(handle, stream))
        return fp

    def _upload(self, handle, indices, stream):
        """Copies the given master parameters into the engine: fp32 contiguous CUDA tensors go through ONE
        mdb_unet_set_params call (argument arrays cached per (index set, storage addresses): the training step re-uploads
        every parameter after every optimiser step); anything else (host tensors, other dtypes) one by one."""
        L = _native.lib()
        indices = tuple(indices)
        params = [self._param(self._names[i]) for i in indices]
        bulk = [k for k, p in enumerate(params) if p.is_cuda and p.dtype == torch.float32 and p.is_contiguous()]
        if bulk:
            key = (tuple(indices[k] for k in bulk), tuple(params[k].data_ptr() for k in bulk))
            cache = getattr(self, "_upload_cache", None)
            if cache is None or cache[0] != key:
                m = len(bulk)
                names = (ctypes.c_char_p * m)(*[self._names[indices[k]].encode() for k in bulk])
                srcs = (ctypes.c_void_p * m)(*key[1])
                numels = (ctypes.c_longlong * m)(*[params[k].numel() for k in bulk])
                cache = self._upload_cache = (key, m, names, srcs, numels)
            _native.check(L.mdb_unet_set_params(handle, cache[1], cache[2], cache[3], cache[4], stream))
        done = set(bulk)
        for k, p in enumerate(params):
            if k in done:
                continue
            src = p.detach().float().contiguous()
            _native.check(L.mdb_unet_set_param(handle, self._names[indices[k]].encode(), _native.ptr(src), src.numel(),
                                               1 if src.is_cuda else 0, stream))
            if src.is_cuda:
                src.record_stream(torch.cuda.current_stream())

    def _train_forward(self, x, labels):
        L = _native.lib()
        B = x.shape[0]
        with torch.cuda.device(x.device):
            self._ensure_train_engine(B, x.device)
            self._train_synced = self._push_parameters(self._train_handle, self._train_synced)
            p = self.dropout if self.training else 0.0
            self._drop_calls += 1
            seed = (torch.initial_seed() * 1000003 + self._drop_calls) & 0xFFFFFFFFFFFFFFFF
            _native.check(L.mdb_unet_set_dropout(self._train_handle, p, seed))
            out = torch.empty_like(x)
            _native.check(L.mdb_unet_forward(self._train_handle, _native.ptr(x), _native.ptr(labels), _native.ptr(out), B,
                                             _native.current_stream()))
        self._pending = (x.data_ptr(), B)
        return out

    def _train_backward(self, x, labels, dout):
        """Engine backward of the LAST forward (its activations live in the engine's arena); gradients go into the flat
        buffer: overwritten when every p.grad is None (after zero_grad), accumulated when they are the buffer's views."""
        L = _native.lib()
        B = x.shape[0]
        if self._pending != (x.data_ptr(), B):
            raise _native.NativeError("backward() must follow the forward() it differentiates: the engine keeps the "
                                      "activations of one forward pass at a time")
        params = [self._param(n) for n in self._trainable]
        none = [p.grad is None for p in params]
        ours = [p.grad is not None and p.grad.data_ptr() == self._grad_views[n].data_ptr() for p, n in zip(params, self._trainable)]
        dout = dout.float().contiguous()
        import torch.distributed as dist
        overlap = (self.reduce_in_backward and self.grad_overlap and dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1
                   and dist.get_backend() == "nccl")
        with torch.cuda.device(x.device):
            if all(none) or all(ours):
                if overlap:
                    self._backward_with_overlapped_allreduce(dout, B, accumulate=not all(none))
                else:
                    _native.check(L.mdb_unet_backward(self._train_handle, _native.ptr(dout), _native.ptr(self._flat_grad),
                                                      self._flat_grad.numel(), B, 0 if all(none) else 1, _native.current_stream()))
                if all(none):
                    for p, n in zip(params, self._trainable):
                        p.grad = self._grad_views[n]
            else:  # gradients owned by someone else: compute into a scratch buffer and add
                tmp = torch.zeros_like(self._flat_grad)
                _native.check(L.mdb_unet_backward(self._train_handle, _native.ptr(dout), _native.ptr(tmp), tmp.numel(), B, 0,
                                                  _native.current_stream()))
                for p, n in zip(params, self._trainable):
                    v = self._grad_views[n]
                    g = tmp[v.storage_offset():v.storage_offset() + v.numel()].view(p.shape)
                    p.grad = g.clone() if p.grad is None else p.grad + g
        self._pending = None

    def allreduce_grads(self):
        """Data-parallel training: the mean of the flat gradient buffer over the ranks (NCCL), replacing the reference's
        nn.DataParallel gather (models/utils.py:95). When the backward pass already launched the bucketed reductions
        (`reduce_in_backward`), this only makes the current stream wait for them; otherwise one blocking all-reduce.
        No-op without an initialised process group."""
        import torch.distributed as dist
        if self._flat_grad is None or not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
            return
        if self._pending_reduce is not None:
            for w in self._pending_reduce:
                w.wait()
            self._pending_reduce = None
            return
        dist.all_reduce(self._flat_grad, op=dist.ReduceOp.SUM)
        self._flat_grad.mul_(1.0 / dist.get_world_size())

    def __del__(self):
        try:
            self.release_engine()
        except Exception:
            pass

    def _fingerprints(self):
        """One kernel over all master parameters -> int64 fingerprints on the host (synchronises)."""
        L = _native.lib()
        params = [self._param(n) for n in self._names]
        key = tuple(p.data_ptr() for p in params)
        if getattr(self, "_fp_key", None) != key:
            dev = params[0].device
            self._fp_ptrs = torch.tensor(key, dtype=torch.int64, device=dev)
            self._fp_numels = torch.tensor([p.numel() for p in params], dtype=torch.int64, device=dev)
            self._fp_out = torch.empty(len(params), dtype=torch.int64, device=dev)
            self._fp_key = key
        _native.check(L.mdb_fingerprint(_native.ptr(self._fp_ptrs), _native.ptr(self._fp_numels), len(params),
                                        _native.ptr(self._fp_out), _native.current_stream()))
        return self._fp_out.cpu()

    def frozen(self):
        """Context manager: the caller promises not to touch the parameters inside (e.g. the sampler loop), so the
        per-call change detection (a 1.5 GB read + a host sync) is skipped."""
        net = self

        class _Frozen:
            def __enter__(self_inner):
                net.sync_parameters()
                net._frozen = True

            def __exit__(self_inner, *exc):
                net._frozen = False

        return _Frozen()

    def sync_parameters(self, force=False):
        """Pushes changed master parameters into the engine and re-derives packed weights / the stem field.
        Changes are detected by content fingerprints, because `p.data[...] = v` (how trainer.py:61-63 writes the mask
        and ema.py copies weights) does not bump autograd's version counters."""
        L = _native.lib()
        if getattr(self, "_frozen", False) and not force:
            return
        fp = self._fingerprints()
        changed = None if (force or self._synced is None) else (fp != self._synced).nonzero().flatten().tolist()
        if changed is not None and not changed:
            return
        stream = _native.current_stream()
        self._upload(self._handle, range(len(self._names)) if changed is None else changed, stream)
        torch.cuda.current_stream().synchronize()
        _native.check(L.mdb_unet_commit(self._handle, stream))
        self._synced = fp

    def forward(self, x, labels):
        if not x.is_cuda:
            raise _native.NativeError("the score network runs only on a CUDA (sm_100a) device; there is no CPU path")
        L = _native.lib()
        x = x.float().contiguous()
        labels = labels.to(device=x.device, dtype=torch.float32).contiguous()
        B = x.shape[0]
        # training path: model.train() + autograd enabled (what step_fn(train=True) sets up, losses.py:104-139 with
        # get_model_fn(train=True)); everything else -- model.eval() or no_grad -- is the inference engine
        if self.training and torch.is_grad_enabled() and any(self._param(n).requires_grad for n in self._trainable):
            out = _ScoreNetFn.apply(self, x, labels, *[self._param(n) for n in self._trainable])
            if self.scale_by_sigma:
                out = out / self.sigmas.to(out.device)[labels.long(), None, None, None, None].float()
            return out
        with torch.cuda.device(x.device):
            self._ensure_engine(B, x.device)
            self.sync_parameters()
            out = torch.empty_like(x)
            _native.check(L.mdb_unet_forward(self._handle, _native.ptr(x), _native.ptr(labels), _native.ptr(out), B,
                                             _native.current_stream()))
        if self.scale_by_sigma:
            out = out / self.sigmas.to(out.device)[labels.long(), None, None, None, None].float()
        return out

    def engine_info(self):
        L = _native.lib()
        fl, ar, ng, ns = ctypes.c_double(), ctypes.c_longlong(), ctypes.c_int(), ctypes.c_int()
        _native.check(L.mdb_unet_info(self._handle, ctypes.byref(fl), ctypes.byref(ar), ctypes.byref(ng), ctypes.byref(ns)))
        return dict(flops_per_sample=fl.value, arena_bytes=ar.value, gemm_launches=ng.value, steps=ns.value,
                    max_batch=self._engine_batch, precision=self.precision)

    def profile(self, x, labels):
        """One profiled forward: [(step name, device ms)]."""
        L = _native.lib()
        B = x.shape[0]
        self._ensure_engine(B, x.device)
        self.sync_parameters()
        out = torch.empty_like(x)
        names = ctypes.create_string_buffer(1 << 16)
        ms = (ctypes.c_float * 1024)()
        n = ctypes.c_int()
        _native.check(L.mdb_unet_profile(self._handle, _native.ptr(x), _native.ptr(labels), _native.ptr(out), B,
                                         _native.current_stream(), names, len(names), ms, 1024, ctypes.byref(n)))
        return list(zip(names.value.decode().strip().split("\n"), [ms[i] for i in range(n.value)]))


@utils.register_model(name="ddpm_res64")
class DDPMRes64(ScoreNet):
    pass


@utils.register_model(name="ddpm_res128")
class DDPMRes128(ScoreNet):
    pass


# configs/res128.py:40 names 'ddpm_res128_v2' although the reference registers only 'ddpm_res128'
# (ddpm_res128.py:41); register both so the stock config works.
utils.register_model(DDPMRes128, name="ddpm_res128_v2")

"""LoRA-wrapped attention projections on the tcgen05 GEMM kernels -- host side.

Mirrors the third-party surface the reference's trainers touch (SURVEY.md section 8 rows a9-a11, b3):

* ``LoraConfig`` / ``add_adapter(unet, cfg)``: what ``unet.add_adapter(LoraConfig(r=..., lora_alpha=...,
  init_lora_weights="gaussian", target_modules=["to_k","to_q","to_v","to_out.0"]))`` does
  (train_online_pso_sdxl_turbo.py:338-345, train_online_pso_sdxl_dmd2.py:361-368,
  train_pso_sdxl_turbo_dreambooth.py:1319-1326).
* ``LoRALinear``: the module peft==0.11.1 puts in place of each target ``nn.Linear``: attributes ``base_layer``,
  ``lora_A[name]``, ``lora_B[name]``, ``scaling[name]``, ``r``, ``lora_alpha``, ``disable_adapters``;
  ``forward(x) = base_layer(x) + lora_B(lora_A(x)) * scaling``.
* ``disable_adapters(unet)`` / ``enable_adapters(unet)``: the policy / frozen-reference switch
  (turbo :790,805; dmd2 :792,807; dreambooth :1897,1918).
* ``PSOAttnProcessor2_0``: diffusers==0.27.0 ``AttnProcessor2_0.__call__`` signature and data flow.
* ``LoRAGradBucket``: every adapter gradient lives in ONE flat fp32 buffer, written in place by the
  weight-gradient kernels (so gradient accumulation costs nothing) and all-reduced with ONE NCCL call
  (the reference: DDP buckets behind accelerator.prepare, turbo :491, sync gate :858).

The forward of a projection is ONE launch (the skinny ``t = s x A^T`` runs as tiles of the same launch as
``y = x W^T + b + t B^T``, one pass over W) where the reference stack issues five; the backward is two (input gradient with
``u = s dy B`` in-launch; both weight gradients).  ``fuse_attention_projections`` stacks q / k / v (k / v) into one such
problem.  There is no PyTorch fallback: a CPU tensor raises.
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass, field
from typing import Iterable, Optional

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib, amp


@dataclass
class LoraConfig:
    """The subset of ``peft.LoraConfig`` the reference passes."""
    r: int = 8
    lora_alpha: int = 8
    init_lora_weights: object = "gaussian"
    target_modules: Iterable[str] = field(default_factory=lambda: ["to_k", "to_q", "to_v", "to_out.0"])
    lora_dropout: float = 0.0


# When a list is installed here, every projection call issues its launches one at a time (psob200 forward_phases /
# backward_phases) and appends (start_event, end_event, flops, algorithmic bytes, role, (M, K, N, r)) per LAUNCH: the
# instrumented pass bench.py uses to attribute device time to the GEMM kernels.  None in normal operation.
_TIMING = None


def set_timing_sink(sink) -> None:
    global _TIMING
    _TIMING = sink


# Weight-gradient side stream.  Nothing downstream of a layer's backward waits for dA / dB (they are read at the optimizer
# boundary), so their two launches can leave the critical path: with ``set_wgrad_stream(True)`` they are issued on a second
# CUDA stream (ordered after the layer's u / dx launches) and joined back once, at the end of the backward pass, by an
# autograd-engine callback.  Works eagerly and under CUDA-graph capture (the fork / join become graph edges).
_WGRAD_SIDE = {"enabled": False, "streams": {}, "pending": {}, "armed": {}}  # armed: device -> id of the backward pass


def set_wgrad_stream(enabled: bool) -> None:
    _WGRAD_SIDE["enabled"] = bool(enabled)


def _wgrad_side_stream(dev: torch.device) -> torch.cuda.Stream:
    st = _WGRAD_SIDE["streams"].get(dev)
    if st is None:
        st = _WGRAD_SIDE["streams"][dev] = torch.cuda.Stream(device=dev)
    return st


def _arm_wgrad_join(dev: torch.device) -> None:
    """Queue (once per backward pass) the callback that makes the caller's stream wait for the side stream and releases
    the operands the side launches were still reading."""
    task = torch._C._current_graph_task_id()
    if _WGRAD_SIDE["armed"].get(dev) == task:
        return
    # a different id means the previous backward pass never reached its callback (it raised): arm again
    _WGRAD_SIDE["armed"][dev] = task

    def join():
        _WGRAD_SIDE["armed"].pop(dev, None)
        torch.cuda.current_stream(dev).wait_stream(_wgrad_side_stream(dev))
        _WGRAD_SIDE["pending"].pop(dev, None)

    torch.autograd.Variable._execution_engine.queue_callback(join)


def _timed_launch(dev, fn, what: str, role: str, flops: float, nbytes: float, shape) -> None:
    """Instrumented pass: ONE kernel launch between two events; appends (ev0, ev1, flops, algorithmic bytes, role, shape)."""
    # external: inside a CUDA-graph capture the records become event-record nodes (timestamps of the last replay)
    ev0, ev1 = torch.cuda.Event(enable_timing=True, external=True), torch.cuda.Event(enable_timing=True, external=True)
    ev0.record()
    with _lib.on_device(dev):
        rc = fn()
    _lib.check(rc, what)
    ev1.record()
    _TIMING.append((ev0, ev1, flops, nbytes, role, shape))


def _ceil8(n: int) -> int:
    return (n + 7) // 8 * 8


class LoRALinear(nn.Module):
    """Drop-in for peft ``lora.Linear`` around a frozen ``nn.Linear`` (one adapter, named like peft's)."""

    def __init__(self, base_layer: nn.Linear, r: int, lora_alpha: int, init_lora_weights="gaussian",
                 adapter_name: str = "default", lora_dtype: torch.dtype = torch.float32):
        super().__init__()
        if r <= 0 or r > 256:
            raise ValueError(f"LoRA rank must be in [1, 256], got {r}")
        self.base_layer = base_layer
        self.in_features, self.out_features = base_layer.in_features, base_layer.out_features
        self.active_adapter = adapter_name
        self.r = {adapter_name: r}
        self.lora_alpha = {adapter_name: lora_alpha}
        self.scaling = {adapter_name: lora_alpha / r}
        dev = base_layer.weight.device
        a = nn.Linear(self.in_features, r, bias=False, device=dev, dtype=lora_dtype)
        b = nn.Linear(r, self.out_features, bias=False, device=dev, dtype=lora_dtype)
        if init_lora_weights == "gaussian":  # peft: normal_(A, std=1/r), zeros_(B)
            nn.init.normal_(a.weight, std=1.0 / r)
        elif init_lora_weights:
            nn.init.kaiming_uniform_(a.weight, a=math.sqrt(5))
        nn.init.zeros_(b.weight)
        self.lora_A = nn.ModuleDict({adapter_name: a})
        self.lora_B = nn.ModuleDict({adapter_name: b})
        self._disable_adapters = False
        self._op_cache = {}  # 16-bit, TMA-friendly copies of the adapter weights, keyed by parameter version
        base_layer.weight.requires_grad_(False)
        if base_layer.bias is not None:
            base_layer.bias.requires_grad_(False)

    # ---- peft surface
    @property
    def disable_adapters(self) -> bool:
        return self._disable_adapters

    def enable_adapters(self, enabled: bool) -> None:
        self._disable_adapters = not enabled

    @property
    def weight(self):
        return self.base_layer.weight

    @property
    def bias(self):
        return self.base_layer.bias

    # ---- operands
    def _operand(self, which: str, dtype: torch.dtype) -> torch.Tensor:
        """The adapter matrix as a 16-bit tensor whose row pitch is a multiple of 16 bytes (A: [r,K]; B: [N,r] in a
        [N, ceil8(r)] buffer).  Re-made only when the parameter changed (optimizer step)."""
        p = (self.lora_A if which == "a" else self.lora_B)[self.active_adapter].weight
        ok = p.dtype == dtype and p.is_contiguous() and p.shape[1] % 8 == 0 and p.data_ptr() % 16 == 0
        if ok:
            return p.detach()
        key = (which, dtype)
        hit = self._op_cache.get(key)
        cols = p.shape[1]
        if hit is None or hit[1] != p.data_ptr() or hit[2].device != p.device:
            buf = torch.zeros(p.shape[0], _ceil8(cols), dtype=dtype, device=p.device)
            hit = [-1, p.data_ptr(), buf[:, :cols]]
            self._op_cache[key] = hit
        if hit[0] != p._version:  # refreshed IN PLACE: the buffer address is stable (CUDA-graph friendly)
            hit[2].copy_(p.detach())
            hit[0] = p._version
        return hit[2]

    def install_operand(self, which: str, dtype: torch.dtype, op: torch.Tensor) -> None:
        """Use ``op`` (the parameter's shape, row pitch a multiple of 16 bytes) as the 16-bit copy of adapter matrix
        ``which``: a view of a flat operand buffer that whoever updates the parameter in place keeps current."""
        p = (self.lora_A if which == "a" else self.lora_B)[self.active_adapter].weight
        self._op_cache[(which, dtype)] = [p._version, p.data_ptr(), op]

    def refresh_operand(self, which: str, dtype: torch.dtype) -> None:
        """Re-make the 16-bit copy of adapter matrix ``which`` even though the parameter's version did not change (a kernel
        wrote the parameter in place)."""
        hit = self._op_cache.get((which, dtype))
        if hit is not None:
            hit[0] = -1
        self._operand(which, dtype)

    def refresh_operands(self) -> None:
        """Bring the 16-bit operand copies up to date with the parameters (call after an optimizer step when the
        forward is replayed from a CUDA graph, where this Python code does not run)."""
        dtype = self.base_layer.weight.dtype
        self._operand("a", dtype)
        self._operand("b", dtype)

    def forward(self, x: torch.Tensor, *args, **kwargs) -> torch.Tensor:
        # the adapter matrices are passed to the autograd function so that the output depends on them (their gradients are
        # accumulated in place by the kernels; the Function returns None for them)
        g = self.__dict__.get("_solo_group")
        if g is None:
            g = self.__dict__["_solo_group"] = LoRAProjectionGroup([self])
        return g(x)


_FLAGS: dict = {}
_IN_LAUNCH_DEPS = {"enabled": True}
_LAUNCH_FLAGS = {"value": 1 if __import__("os").environ.get("PSOB200_PROGRAMMATIC_LAUNCH", "0") == "1" else 0}


def set_deterministic_wgrad(enabled: bool) -> None:
    """Bit-reproducible adapter gradients (psob200_lora_group_args.launch_flags bit 1): the dA / dB reductions are not split
    over CTAs, so the fp32 atomic accumulation has exactly one contribution per element and launch.  Slower weight-gradient
    launches (they are off the critical path with ``set_wgrad_stream(True)``)."""
    _LAUNCH_FLAGS["value"] = (_LAUNCH_FLAGS["value"] & ~2) | (2 if enabled else 0)


def set_programmatic_launch(enabled: bool) -> None:
    """A/B switch (psob200_lora_group_args.launch_flags bit 0): launch the projection kernels with programmatic stream
    serialization, so that their launch latency and prologue overlap the tail of the preceding kernel on the stream."""
    _LAUNCH_FLAGS["value"] = (_LAUNCH_FLAGS["value"] & ~1) | (1 if enabled else 0)


def set_in_launch_dependencies(enabled: bool) -> None:
    """A/B switch: False issues t / u as launches of their own (programmatic dependent launch overlaps them with the main
    pass, as in round 1) instead of as tiles of the main launch.  Results are bit-identical."""
    _IN_LAUNCH_DEPS["enabled"] = bool(enabled)


def _flags_workspace(dev: torch.device) -> torch.Tensor:
    """Zeroed int32 scratch for the in-launch dependencies of the fused projection launches (psob200_lora_group_args.flags):
    one per (device, stream) -- launches on a stream are ordered and every launch leaves it zeroed."""
    key = (dev, torch.cuda.current_stream(dev).cuda_stream)
    ws = _FLAGS.get(key)
    if ws is None:
        ws = _FLAGS[key] = torch.zeros(8192, dtype=torch.int32, device=dev)
    return ws


class LoRAProjectionGroup:
    """G LoRA-wrapped projections that read the SAME input, run as one stacked problem (psob200_lora_group_*): attention
    to_q / to_k / to_v (G = 3), cross-attention to_k / to_v (G = 2), or a single ``LoRALinear`` (G = 1).

    The frozen weights of the members become views of ONE [G N, K] matrix (their values are unchanged; ``layer.weight`` still
    works).  The adapters are consumed stacked as well: when the members' 16-bit operand copies (and fp32 gradient targets) sit
    next to each other in memory -- they do once ``LoRAGradBucket`` / ``FusedLoRAOptimizer`` laid the parameters out in
    ``lora_parameters()`` order -- they are used in place; otherwise the group keeps private stacked copies."""

    def __init__(self, layers):
        layers = list(layers)
        l0 = layers[0]
        for l in layers[1:]:
            if (l.in_features, l.out_features) != (l0.in_features, l0.out_features) or l.r != l0.r or l.scaling != l0.scaling \
                    or l.base_layer.weight.dtype != l0.base_layer.weight.dtype or l.active_adapter != l0.active_adapter:
                raise ValueError("stacked projections must have the same shape, rank, scaling and dtype")
        if len(layers) > 1 and any(l.base_layer.bias is not None for l in layers):
            raise ValueError("stacked projections must not have a bias (attention q / k / v have none)")
        self.layers = layers
        self.G = len(layers)
        self.K, self.N = l0.in_features, l0.out_features
        r = l0.r[l0.active_adapter]
        # stride of the G column groups of the stacked t / u: the rank itself, or -- when it is not a multiple of 8 -- the rank
        # rounded up to 8 (the groups must start on 16-byte boundaries): lora_a is then stacked with zero rows in between
        self.r_stride = r if (self.G == 1 or r % 8 == 0) else _ceil8(r)
        self._op = {}     # which -> [versions, stacked 16-bit buffer]
        self._grad = {}   # which -> stacked fp32 gradient buffer (only without a flat bucket)
        if self.G > 1:
            w = torch.cat([l.base_layer.weight.detach() for l in layers], dim=0).contiguous()
            for g, l in enumerate(layers):
                l.base_layer.weight.data = w[g * self.N:(g + 1) * self.N]
            self.weight = w
        else:
            self.weight = None

    @property
    def name(self):
        return self.layers[0].active_adapter

    def stacked_weight(self) -> torch.Tensor:
        if self.G == 1:
            return self.layers[0].base_layer.weight
        ws = [l.base_layer.weight.detach() for l in self.layers]
        if self._adjacent(ws):  # views of this group's buffer -- or of a bigger one (CrossKVBank stacks many groups)
            return ws[0].as_strided((self.G * self.N, self.K), (self.K, 1))
        w = torch.cat(ws, dim=0).contiguous()  # model.to(...) moved the members
        for g, l in enumerate(self.layers):
            l.base_layer.weight.data = w[g * self.N:(g + 1) * self.N]
        self.weight = w
        return w

    def _adjacent(self, tensors) -> bool:
        t0 = tensors[0]
        step = t0.numel() * t0.element_size()
        base = t0.untyped_storage().data_ptr()  # slices of ONE buffer (the flat layout), not neighbours by allocator luck
        return all(t.is_contiguous() and t.untyped_storage().data_ptr() == base and t.data_ptr() == t0.data_ptr() + g * step
                   for g, t in enumerate(tensors))

    def stacked_operand(self, which: str, dtype: torch.dtype) -> torch.Tensor:
        """[G r_stride, K] (which = "a") or [G N, r] ("b") 16-bit, row pitch a multiple of 8 elements."""
        ops = [l._operand(which, dtype) for l in self.layers]
        if self.G == 1:
            return ops[0]
        r = ops[0].shape[0] if which == "a" else ops[0].shape[1]
        packed = self.r_stride == r
        if packed and self._adjacent(ops) and ops[0].stride(0) == ops[0].shape[1]:
            return ops[0].as_strided((self.G * ops[0].shape[0], ops[0].shape[1]), (ops[0].shape[1], 1))
        # private stacked copy (members not adjacent, or a rank that needs padding), refreshed IN PLACE when a member changed:
        # stable address (CUDA-graph friendly); FusedLoRAOptimizer.step() calls refresh_operands() for such groups
        params = [(l.lora_A if which == "a" else l.lora_B)[l.active_adapter].weight for l in self.layers]
        vers = tuple((p.data_ptr(), p._version) for p in params)
        hit = self._op.get((which, dtype))
        if hit is None or hit[1].device != ops[0].device:
            if which == "a":
                buf = torch.zeros(self.G * self.r_stride, ops[0].shape[1], dtype=dtype, device=ops[0].device)
            else:
                buf = torch.zeros(self.G * ops[0].shape[0], _ceil8(r), dtype=dtype, device=ops[0].device)
            hit = [None, buf]
            self._op[(which, dtype)] = hit
        if hit[0] != vers:
            rows = self.r_stride if which == "a" else ops[0].shape[0]
            src = [p.detach() for p in params]
            if self._adjacent(src):
                # the members' parameters are consecutive slices of one flat buffer (FusedLoRAOptimizer / LoRAGradBucket built from
                # lora_parameters()): ONE strided, converting copy instead of G (a cross-attention bank stacks 120 projections)
                s0 = src[0]
                stacked = s0.as_strided((self.G, s0.shape[0], s0.shape[1]), (s0.numel(), s0.shape[1], 1))
                hit[1].view(self.G, rows, hit[1].shape[1])[:, :s0.shape[0], :s0.shape[1]].copy_(stacked)
            else:
                for g, o in enumerate(ops):
                    hit[1][g * rows:g * rows + o.shape[0], :o.shape[1]].copy_(o)
            hit[0] = vers
        return hit[1] if which == "a" else hit[1][:, :r]

    def has_private_operands(self) -> bool:
        return bool(self._op)

    def refresh_operands(self) -> None:
        dtype = self.layers[0].base_layer.weight.dtype
        self.stacked_operand("a", dtype)
        self.stacked_operand("b", dtype)

    def refresh_private_operands(self) -> None:
        """Re-stack the private copies, if the group keeps any, even though no member's version changed (a kernel wrote
        the parameters in place)."""
        if self._op:
            for hit in self._op.values():
                hit[0] = None
            self.refresh_operands()

    def stacked_grad(self, which: str) -> torch.Tensor:
        """fp32 accumulation target [G r, K] / [G N, r]: the members' slices of the flat bucket when they are adjacent, else
        a private stacked buffer the members' ``.grad`` become views of."""
        params = [(l.lora_A if which == "a" else l.lora_B)[l.active_adapter].weight for l in self.layers]
        if any(p.dtype != torch.float32 for p in params):
            raise _lib.Psob200Error("stacked projections train fp32 adapter parameters (the shipped mixed-precision recipes)")
        if self.G == 1:
            return _grad_buffer(params[0])
        views = [getattr(p, "_psob200_grad_view", None) for p in params]
        if all(v is not None for v in views):
            if not self._adjacent(views):
                raise _lib.Psob200Error("the gradient slices of stacked projections are not adjacent in the flat bucket: build "
                                        "LoRAGradBucket / FusedLoRAOptimizer from lora.lora_parameters(model) AFTER "
                                        "lora.fuse_attention_projections(model)")
            for p in params:
                _grad_buffer(p)  # re-attach p.grad / refuse foreign tensors
            v0 = views[0]
            return v0.as_strided((self.G * v0.shape[0], v0.shape[1]), (v0.shape[1], 1))
        buf = torch.zeros(self.G * params[0].shape[0], params[0].shape[1], dtype=torch.float32, device=params[0].device)
        rows = params[0].shape[0]
        for g, p in enumerate(params):
            v = buf[g * rows:(g + 1) * rows]
            if p.grad is not None:
                v.copy_(p.grad)
            p.grad = v
            p._psob200_grad_view = v
        self._grad[which] = buf
        return buf

    def __call__(self, x: torch.Tensor):
        """Returns the G projections of ``x`` (views of one [.., G N] buffer)."""
        params = []
        for l in self.layers:
            params += [l.lora_A[l.active_adapter].weight, l.lora_B[l.active_adapter].weight]
        return _LoraGroupFn.apply(x, self, torch.is_grad_enabled(), *params)


class _LoraGroupFn(torch.autograd.Function):
    """psob200_lora_group_forward / _backward.  Gradients of the adapter matrices are ACCUMULATED IN PLACE into
    ``param.grad`` (fp32 views of the flat bucket when one is attached), so autograd receives only ``dx``."""

    @staticmethod
    def forward(ctx, x: torch.Tensor, group: LoRAProjectionGroup, grad_mode: bool, *params):
        want_wgrad = grad_mode and params[0].requires_grad  # False under no_grad (the frozen-reference pass)
        x2, y, tt, enabled = _group_forward_launch(x, group, want_wgrad)
        G, N = group.G, group.N
        ctx.group, ctx.enabled, ctx.x_shape, ctx.x_dtype, ctx.want_wgrad = group, enabled, x.shape, x.dtype, want_wgrad and enabled
        ctx.save_for_backward(x2, tt)
        y = y.view(*x.shape[:-1], G * N)
        if G == 1:
            return y
        return tuple(y[..., g * N:(g + 1) * N] for g in range(G))

    @staticmethod
    def backward(ctx, *dys):
        return _group_backward(ctx, dys) + (None,) * (2 * ctx.group.G)


def _group_forward_launch(x: torch.Tensor, group: LoRAProjectionGroup, want_wgrad: bool):
    """psob200_lora_group_forward for ``group``: returns (x as the [M, K] operand, y [M, G N], tt or None, adapters enabled)."""
    l0 = group.layers[0]
    w = group.stacked_weight()
    dev = _lib.require_cuda(x, w)
    dtype = w.dtype
    if dtype not in (torch.bfloat16, torch.float16):
        raise _lib.Psob200Error(f"the tcgen05 LoRA path needs bf16/fp16 base weights, got {dtype}")
    G, K, N = group.G, group.K, group.N
    if x.shape[-1] != K:
        raise _lib.Psob200Error(f"input feature size {x.shape[-1]} != in_features {K}")
    x2 = x.detach().reshape(-1, K)
    if x2.dtype != dtype:
        x2 = x2.to(dtype)
    if not x2.is_contiguous() or x2.data_ptr() % 16:
        x2 = x2.contiguous()
    if K % 8 or w.stride(0) != K or w.data_ptr() % 16:
        raise _lib.Psob200Error("base weight must be contiguous with in_features a multiple of 8")
    M = x2.shape[0]
    enabled = not l0._disable_adapters
    if any(l._disable_adapters != l0._disable_adapters for l in group.layers):
        raise _lib.Psob200Error("stacked projections must be enabled / disabled together")
    name = l0.active_adapter
    r = l0.r[name]
    rs = group.r_stride
    a = _lib.LoraGroupArgs()
    y = torch.empty(M, G * N, dtype=dtype, device=dev)
    a.x, a.ldx, a.w, a.ldw, a.y, a.ldy = x2.data_ptr(), K, w.data_ptr(), K, y.data_ptr(), G * N
    bias = l0.base_layer.bias if G == 1 else None
    if bias is not None:
        a.bias, a.bias_dtype = bias.data_ptr(), _lib.dtype_code(bias)
    a.M, a.K, a.N, a.r, a.G, a.r_stride = M, K, N, r, G, rs
    a.dtype = _lib.dtype_code(x2)
    a.adapters_enabled = int(enabled)
    a.launch_flags = _LAUNCH_FLAGS["value"]
    want_wgrad = enabled and want_wgrad
    t = tt = None
    fl_t = by_t = 0.0
    if enabled:
        la, lb = group.stacked_operand("a", dtype), group.stacked_operand("b", dtype)
        gr8 = _ceil8(G * rs)
        t = torch.empty(M, gr8, dtype=dtype, device=dev)
        a.lora_a, a.lda, a.lora_b, a.ldb = la.data_ptr(), la.stride(0), lb.data_ptr(), lb.stride(0)
        a.t, a.ldt = t.data_ptr(), gr8
        a.scaling = float(l0.scaling[name])
        if want_wgrad:
            tt = torch.empty(G * rs, _ceil8(M), dtype=dtype, device=dev)
            a.tt, a.ldtt = tt.data_ptr(), tt.stride(0)
        if _IN_LAUNCH_DEPS["enabled"]:
            ws = _flags_workspace(dev)  # t becomes tiles of the same launch as y
            a.flags, a.flags_len = ws.data_ptr(), ws.numel()
        fl_t = 2.0 * M * G * r * K
        by_t = 2 * (G * r * K + M * G * r * (2 if tt is not None else 1))
    if _TIMING is None:
        _lib.launch(dev, "psob200_lora_group_forward", C.byref(a), _lib.current_stream(dev))
    else:  # instrumented pass: the same launch between its own pair of events
        role = ("y = x W^T + t B^T (t = s x A^T as tiles of the same launch)" if enabled else "y = x W^T (frozen reference)")
        _timed_launch(dev, lambda: _lib.lib().psob200_lora_group_forward(C.byref(a), _lib.current_stream(dev)),
                      "psob200_lora_group_forward", role, 2.0 * M * G * N * (K + (r if enabled else 0)) + fl_t,
                      2 * (M * K + G * N * K + M * G * N + (G * N * r if enabled else 0)) + by_t, (M, K, G * N, r if enabled else 0))
    return x2, y, tt, enabled


def _group_backward(ctx, dys):
    """psob200_lora_group_backward for the node ``ctx`` (``ctx.group``, saved (x2, tt)): returns (dx, None, None)."""
    group: LoRAProjectionGroup = ctx.group
    x2, tt = ctx.saved_tensors
    l0 = group.layers[0]
    w = group.stacked_weight()
    dev, dtype = w.device, w.dtype
    G, K, N = group.G, group.K, group.N
    M = x2.shape[0]
    name = l0.active_adapter
    r = l0.r[name]
    a = _lib.LoraGroupArgs()
    dy2 = []
    for g in range(G):
        d = dys[g].reshape(-1, N)
        if d.dtype != dtype:
            d = d.to(dtype)
        if d.stride(1) != 1 or d.stride(0) % 8 or d.data_ptr() % 16:
            d = d.contiguous()
        dy2.append(d)
        a.dy[g], a.lddy[g] = d.data_ptr(), d.stride(0)
    a.w, a.ldw, a.x, a.ldx = w.data_ptr(), K, x2.data_ptr(), K
    rs = group.r_stride
    a.M, a.K, a.N, a.r, a.G, a.r_stride = M, K, N, r, G, rs
    a.dtype = _lib.dtype_code(dy2[0])
    a.adapters_enabled = int(ctx.enabled)
    a.launch_flags = _LAUNCH_FLAGS["value"]
    dx = None
    if ctx.needs_input_grad[0]:
        dx = torch.empty(M, K, dtype=dtype, device=dev)
        a.dx, a.lddx = dx.data_ptr(), K
    keep = []
    wg = False
    if ctx.enabled:
        la, lb = group.stacked_operand("a", dtype), group.stacked_operand("b", dtype)
        a.lora_a, a.lda, a.lora_b, a.ldb = la.data_ptr(), la.stride(0), lb.data_ptr(), lb.stride(0)
        a.scaling = float(l0.scaling[name])
        gr8 = _ceil8(G * rs)
        u = torch.empty(M, gr8, dtype=dtype, device=dev)
        a.u, a.ldu = u.data_ptr(), gr8
        keep.append(u)
        if _IN_LAUNCH_DEPS["enabled"]:
            ws = _flags_workspace(dev)
            a.flags, a.flags_len = ws.data_ptr(), ws.numel()
        if ctx.want_wgrad:
            ga, gb = group.stacked_grad("a"), group.stacked_grad("b")
            ut = torch.empty(G * rs, _ceil8(M), dtype=dtype, device=dev)
            a.ut, a.ldut = ut.data_ptr(), ut.stride(0)
            a.tt, a.ldtt = tt.data_ptr(), tt.stride(0)
            a.d_lora_a, a.ld_da = ga.data_ptr(), ga.stride(0)
            a.d_lora_b, a.ld_db = gb.data_ptr(), gb.stride(0)
            keep += [ut, ga, gb]
            wg = True
    if dx is not None or wg:
        side = _WGRAD_SIDE["enabled"] and wg and _TIMING is None
        if _TIMING is not None:  # instrumented pass: one launch at a time, each between its own pair of events
            eb = 2
            if dx is not None or wg:
                fl = (2.0 * M * K * G * N if dx is not None else 0.0) + (2.0 * M * G * r * (N + (K if dx is not None else 0)) if ctx.enabled else 0.0)
                by = eb * (M * G * N + (G * N * K + M * K if dx is not None else 0) + ((G * N * r + G * r * K + M * G * r * (2 if wg else 1)) if ctx.enabled else 0))
                role = ("dx = dy W + u A (u = s dy B as tiles of the same launch)" if dx is not None else "u = s dy B")
                a.backward_phases = 3
                _timed_launch(dev, lambda: _lib.lib().psob200_lora_group_backward(C.byref(a), _lib.current_stream(dev)),
                              "psob200_lora_group_backward", role, fl, by, (M, K, G * N, r if ctx.enabled else 0))
            if wg:
                a.backward_phases = 12
                _timed_launch(dev, lambda: _lib.lib().psob200_lora_group_backward(C.byref(a), _lib.current_stream(dev)),
                              "psob200_lora_group_backward", "dA += u^T x ; dB += dy^T t (one launch)",
                              2.0 * M * G * r * (K + N), eb * (M * K + M * G * N + 2 * M * G * r) + 4 * G * r * (K + N),
                              (M, K, G * N, r))
        else:
            if side:
                a.backward_phases = 3  # PSOB200_BWD_INPUT_GRAD: u (+ ut), dx
            _lib.launch(dev, "psob200_lora_group_backward", C.byref(a), _lib.current_stream(dev))
        if side:
            st = _wgrad_side_stream(dev)
            st.wait_stream(torch.cuda.current_stream(dev))
            a.backward_phases = 12  # PSOB200_BWD_WEIGHT_GRAD: dA, dB
            _lib.launch(dev, "psob200_lora_group_backward", C.byref(a), st.cuda_stream)
            _WGRAD_SIDE["pending"].setdefault(dev, []).append((x2, tt, dy2, keep))  # alive until the join
            keep = []
            _arm_wgrad_join(dev)
    del keep
    if dx is not None:
        dx = dx.view(ctx.x_shape)
        if dx.dtype != ctx.x_dtype:
            dx = dx.to(ctx.x_dtype)
    return (dx, None, None)


def _grad_buffer(p: torch.nn.Parameter) -> torch.Tensor:
    """fp32 accumulation target of a LoRA parameter: ``p.grad`` itself for fp32 parameters (a view of the flat
    bucket once ``LoRAGradBucket`` is attached), else a side buffer ``p.grad32`` folded in by ``finalize_grads``."""
    view = getattr(p, "_psob200_grad_view", None)  # set by LoRAGradBucket: this parameter's slice of the flat buffer
    if p.dtype == torch.float32:
        if view is not None:
            if p.grad is None:  # zero_grad(set_to_none=True) / `p.grad = None` detached it: the slice is still the target
                p.grad = view
            elif p.grad.data_ptr() != view.data_ptr():
                raise _lib.Psob200Error("param.grad was replaced by a tensor that is not this parameter's view of the flat LoRA "
                                        "gradient bucket: the exchange / clip / optimizer would read stale zeros.  Zero "
                                        "gradients with LoRAGradBucket.zero_grad() / FusedLoRAOptimizer.zero_grad().")
            return view
        if p.grad is None:
            p.grad = torch.zeros_like(p)
        return p.grad
    if view is not None:
        return view
    g = getattr(p, "grad32", None)
    if g is None:
        g = torch.zeros(p.shape, dtype=torch.float32, device=p.device)
        p.grad32 = g
    return g


# ----------------------------------------------------------------------------------------------- model-level API
def lora_layers(model: nn.Module):
    return [m for m in model.modules() if isinstance(m, LoRALinear)]


def add_adapter(model: nn.Module, config: LoraConfig, adapter_name: str = "default",
                lora_dtype: torch.dtype = torch.float32) -> list:
    """``unet.add_adapter(cfg)``: wrap every ``nn.Linear`` whose qualified name ends with one of
    ``config.target_modules`` (peft matches by suffix, so "to_out.0" hits ``...attn{1,2}.to_out.0`` only).
    ``lora_dtype=float32`` is what the shipped fp16 recipes train (turbo :346-350); pass the base dtype to mimic the
    bf16 recipes, where peft leaves the adapters in the base dtype."""
    targets = list(config.target_modules)
    wrapped = []
    for parent_name, parent in list(model.named_modules()):
        for child_name, child in list(parent.named_children()):
            full = f"{parent_name}.{child_name}" if parent_name else child_name
            if isinstance(child, nn.Linear) and any(full == t or full.endswith("." + t) for t in targets):
                new = LoRALinear(child, config.r, config.lora_alpha, config.init_lora_weights, adapter_name, lora_dtype)
                setattr(parent, child_name, new)
                wrapped.append(new)
    if not wrapped:
        raise ValueError(f"no nn.Linear matches target_modules={targets}")
    return wrapped


def disable_adapters(model: nn.Module) -> None:
    for m in lora_layers(model):
        m.enable_adapters(False)


def enable_adapters(model: nn.Module) -> None:
    for m in lora_layers(model):
        m.enable_adapters(True)


def fuse_attention_projections(model: nn.Module) -> int:
    """Stack the LoRA-wrapped projections that share their input: ``to_q / to_k / to_v`` of every self-attention module become
    one ``LoRAProjectionGroup`` (G = 3), ``to_k / to_v`` of every cross-attention module one (G = 2).  ``PSOAttnProcessor2_0``
    then issues one launch per group (forward), one for the input gradient and one for the weight gradients (backward) instead of
    2 + 4 per projection.  Call it after ``add_adapter`` and BEFORE building ``LoRAGradBucket`` / ``FusedLoRAOptimizer`` (the flat
    layout follows ``lora_parameters()``, which keeps a group's matrices adjacent).  Modules whose projections have biases or
    different shapes keep the per-projection path; a rank that is not a multiple of 8 is stacked with padded private operand
    copies (refreshed by ``FusedLoRAOptimizer.step()`` / ``refresh_operands``).  Returns the number of groups."""
    n = 0
    for m in model.modules():
        q, k, v = (getattr(m, a, None) for a in ("to_q", "to_k", "to_v"))
        if not all(isinstance(t, LoRALinear) for t in (q, k, v)) or "_psob200_groups" in m.__dict__:
            continue
        if any(t.base_layer.bias is not None for t in (q, k, v)):
            continue
        same = lambda a, b: (a.in_features, a.out_features, a.r, a.scaling) == (b.in_features, b.out_features, b.r, b.scaling)
        cross = getattr(m, "is_cross_attention", None)  # diffusers' Attention says so; otherwise: k / v read another width than q
        if cross is None:
            cross = not same(q, k)
        if not cross and same(k, v) and same(q, k):
            members, key = [q, k, v], "qkv"
        elif same(k, v):
            members, key = [k, v], "kv"
        else:
            continue
        group = LoRAProjectionGroup(members)
        for t in members:
            t.__dict__["_psob200_group"] = group
        m.__dict__["_psob200_groups"] = {key: group}
        n += 1
    return n


# ---- the k / v projections of EVERY cross-attention layer in one launch ---------------------------------------------------
# They all read the prompt embeddings and nothing else (the trainers pass one ``encoder_hidden_states`` to every block: T:775-805,
# TP:136): 70 launches per UNet forward with M = 2B x 77 rows -- 25-50 tiles on 148 SMs, 24-34 us each, on the blocks' critical
# path.  ``fuse_cross_attention_kv(unet)`` stacks them per shape (SDXL: 20 projections of width 640, 120 of width 1280) into
# forward-only groups whose ONE launch at the start of the forward writes every block's k and v; each block's processor picks its
# columns up.  The backward stays per layer (the gradients arrive block by block): every block gets its own autograd node over
# views of the bank's results, with the same psob200_lora_group_backward launches as before.


class _Precomputed:
    """Forward results of one stacked group, produced by a bank launch (kept out of autograd's sight)."""

    def __init__(self, x2, y, tt, enabled):
        self.x2, self.y, self.tt, self.enabled = x2, y, tt, enabled


class _PrecomputedGroupFn(torch.autograd.Function):
    """Autograd node of ONE stacked group whose forward was part of a ``CrossKVBank`` launch: the forward hands out views, the
    backward is the group's own ``psob200_lora_group_backward``."""

    @staticmethod
    def forward(ctx, x: torch.Tensor, group: LoRAProjectionGroup, pre: _Precomputed, *params):
        ctx.group, ctx.enabled, ctx.x_shape, ctx.x_dtype = group, pre.enabled, x.shape, x.dtype
        ctx.want_wgrad = pre.enabled and pre.tt is not None
        ctx.save_for_backward(pre.x2, pre.tt)
        N = group.N
        y = pre.y.view(*x.shape[:-1], group.G * N)
        return tuple(y[..., g * N:(g + 1) * N] for g in range(group.G))

    @staticmethod
    def backward(ctx, *dys):
        return _group_backward(ctx, dys) + (None,) * (2 * ctx.group.G)


class CrossKVBank:
    """The ``to_k`` / ``to_v`` groups of cross-attention layers of one shape, stacked for the forward."""

    def __init__(self, members):
        self.members = list(members)  # (attention module, its LoRAProjectionGroup "kv")
        layers = [l for _, g in self.members for l in g.layers]
        self.all = LoRAProjectionGroup(layers)  # re-homes the frozen weights into ONE [sum G N, K] matrix
        for _, g in self.members:
            g.weight = None  # (its members are views of the bank's matrix now: stacked_weight() finds them adjacent)
        for l in layers:
            l.__dict__["_psob200_bank"] = self

    def __call__(self, enc: torch.Tensor, state: Optional[dict] = None) -> None:
        """``state["live"]`` is cleared when the forward that made these entries returns: afterwards only the recomputation of a
        gradient-checkpointed block (inside a backward pass) may still use them -- never a later, unrelated call with the same tensor."""
        state = state if state is not None else {"live": True}
        l0 = self.all.layers[0]
        want = torch.is_grad_enabled() and l0.lora_A[l0.active_adapter].weight.requires_grad
        x2, y, tt, enabled = _group_forward_launch(enc, self.all, want)
        N, rs = self.all.N, self.all.r_stride
        col = row = 0
        for attn, g in self.members:
            ys = y[:, col:col + g.G * N]
            if want and enabled:
                params = []
                for l in g.layers:
                    params += [l.lora_A[l.active_adapter].weight, l.lora_B[l.active_adapter].weight]
                pre = _Precomputed(x2, ys, tt[row:row + g.G * rs] if tt is not None else None, enabled)
                key, value = _PrecomputedGroupFn.apply(enc, g, pre, *params)
            else:
                yv = ys.view(*enc.shape[:-1], g.G * N)
                key, value = yv[..., :N], yv[..., N:]
            attn.__dict__["_psob200_kv"] = (enc, key, value, state)
            col += g.G * N
            row += g.G * rs


def fuse_cross_attention_kv(unet: nn.Module) -> int:
    """Stack the cross-attention ``to_k`` / ``to_v`` groups of ``unet`` (made by ``fuse_attention_projections``) into
    ``CrossKVBank``s, one per (in_features, out_features, rank, scaling, dtype), and install the forward pre-hook that runs them on
    the ``encoder_hidden_states`` the UNet is called with (third positional argument or keyword, diffusers 0.27.0
    ``UNet2DConditionModel.forward``).  Call it after ``fuse_attention_projections`` and BEFORE building ``LoRAGradBucket`` /
    ``FusedLoRAOptimizer`` (``lora_parameters()`` then lays a bank's matrices out next to each other, so that the stacked adapter
    operands are views of the flat buffers instead of copies).  Modules with ``norm_cross`` keep their in-place projections, as do
    calls with another ``encoder_hidden_states``; the recomputation of a gradient-checkpointed block picks up the same k / v as its
    first pass.  Returns the number of banks."""
    if "_psob200_kv_banks" in unet.__dict__:
        return len(unet.__dict__["_psob200_kv_banks"])
    by_shape = {}
    for m in unet.modules():
        groups = m.__dict__.get("_psob200_groups")
        if not groups or "kv" not in groups or getattr(m, "norm_cross", None):
            continue
        g = groups["kv"]
        l0 = g.layers[0]
        key = (g.K, g.N, l0.r[l0.active_adapter], l0.scaling[l0.active_adapter], l0.base_layer.weight.dtype, l0.base_layer.weight.device)
        by_shape.setdefault(key, []).append((m, g))
    banks = [CrossKVBank(members) for members in by_shape.values() if len(members) > 1]
    unet.__dict__["_psob200_kv_banks"] = banks

    live = []

    def hook(module, args, kwargs):
        enc = kwargs.get("encoder_hidden_states", args[2] if len(args) > 2 else None)
        if torch.is_tensor(enc) and enc.is_cuda:
            state = {"live": True}
            live.append(state)
            for bank in banks:
                if enc.shape[-1] == bank.all.K:
                    bank(enc, state)
        return None

    def done(module, args, output):
        while live:
            live.pop()["live"] = False
        return None

    if banks:
        unet.__dict__["_psob200_kv_hook"] = (unet.register_forward_pre_hook(hook, with_kwargs=True), unet.register_forward_hook(done))
    return len(banks)


def projection_groups(model: nn.Module) -> list:
    out = [g for m in model.modules() for g in m.__dict__.get("_psob200_groups", {}).values()]
    return out + [b.all for b in model.__dict__.get("_psob200_kv_banks", [])]


def refresh_operands(model: nn.Module) -> None:
    for m in lora_layers(model):
        m.refresh_operands()
    for g in projection_groups(model):
        g.refresh_operands()


def lora_parameters(model: nn.Module):
    """The trainable adapter matrices in FLAT-LAYOUT order: per projection ``A, B``; for a stacked group all ``A`` of its
    members, then all ``B``; for a ``CrossKVBank`` all ``A`` of all its groups, then all ``B`` -- so that a group's (a bank's)
    matrices are adjacent in the flat buffers built from this list."""
    out, seen = [], set()
    for m in lora_layers(model):
        bank = m.__dict__.get("_psob200_bank")
        if bank is not None:  # all A of the bank (block by block: a block's k / v stay adjacent), then all B
            if id(bank) not in seen:
                seen.add(id(bank))
                out += [l.lora_A[l.active_adapter].weight for l in bank.all.layers]
                out += [l.lora_B[l.active_adapter].weight for l in bank.all.layers]
            continue
        g = m.__dict__.get("_psob200_group")
        if g is None:
            n = m.active_adapter
            out += [m.lora_A[n].weight, m.lora_B[n].weight]
        elif id(g) not in seen:
            seen.add(id(g))
            out += [l.lora_A[l.active_adapter].weight for l in g.layers]
            out += [l.lora_B[l.active_adapter].weight for l in g.layers]
    return out


class LoRAGradBucket:
    """All adapter gradients in one flat fp32 buffer.

    ``param.grad`` of every fp32 adapter matrix becomes a view of ``self.flat``; the dA / dB kernels accumulate
    into those views directly.  ``all_reduce()`` is the data-parallel exchange of the whole training step: one
    collective over the flat buffer, averaged over ranks (what DDP does for the reference, bucket by bucket).
    ``clip_grad_norm_`` is accelerate's ``clip_grad_norm_`` (turbo :859) on the flat buffer: one norm, one scale."""

    def __init__(self, params: Iterable[torch.nn.Parameter], align: int = 8, allocator=None):
        self.params = [p for p in params if p.requires_grad]
        if not self.params:
            raise ValueError("no trainable LoRA parameters")
        dev = self.params[0].device
        sizes = [(p.numel() + align - 1) // align * align for p in self.params]  # every view (also a 16-bit twin) 16-byte aligned
        # allocator(n, device) -> zeroed fp32 tensor of n elements: lets the buffer live in symmetric memory (SymmetricGradExchange)
        self.flat = (torch.zeros(sum(sizes), dtype=torch.float32, device=dev) if allocator is None
                     else allocator(sum(sizes), dev))
        self.views, self.offsets = [], []
        off = 0
        for p, n in zip(self.params, sizes):
            v = self.flat[off:off + p.numel()].view(p.shape)
            self.offsets.append(off)
            off += n
            self.views.append(v)
            p._psob200_grad_view = v  # _grad_buffer re-attaches it if the trainer sets p.grad = None
            if p.dtype == torch.float32:
                p.grad = v
            else:
                p.grad32 = v

    def zero_(self) -> None:
        self.flat.zero_()

    def zero_grad(self, set_to_none: bool = False) -> None:
        """``optimizer.zero_grad()`` for the flat bucket: zeroes IN PLACE and keeps every ``param.grad`` a view of the flat
        buffer (``set_to_none`` is accepted for signature compatibility and ignored: detaching the views would make the
        exchange and the optimizer read zeros)."""
        self.flat.zero_()
        for p, v in zip(self.params, self.views):
            if p.dtype == torch.float32:
                p.grad = v

    def all_reduce(self, group=None, async_op: bool = False):
        """Average the flat gradient over the data-parallel ranks with ONE collective."""
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
            return None
        op = dist.ReduceOp.AVG if dist.get_backend(group) == "nccl" else dist.ReduceOp.SUM
        work = dist.all_reduce(self.flat, op=op, group=group, async_op=async_op)
        if op == dist.ReduceOp.SUM:
            if async_op:
                work.wait()
                work = None
            self.flat.div_(dist.get_world_size(group))
        return work

    def clip_grad_norm_(self, max_norm: float) -> torch.Tensor:
        norm = torch.linalg.vector_norm(self.flat)
        self.flat.mul_(torch.clamp(max_norm / (norm + 1e-6), max=1.0))
        return norm

    def finalize_grads(self) -> None:
        """For 16-bit adapter parameters: publish the fp32 accumulators as ``param.grad`` in the parameter dtype."""
        for p, v in zip(self.params, self.views):
            if p.dtype != torch.float32:
                p.grad = v.to(p.dtype)


class SymmetricGradExchange:
    """The flat LoRA gradient in NVLink symmetric memory, exchanged by ONE kernel of ours per rank instead of an NCCL call.

    ``torch.distributed._symmetric_memory`` is used only as plumbing (allocation, the multicast mapping, the cross-rank
    barrier on the stream).  ``exchange()`` = barrier, ``psob200_flat_allreduce_sumsq`` (in-switch reduction of this rank's
    slice with ``multimem.ld_reduce``, mean, broadcast to every rank with ``multimem.st``, the slice's sum of squares for
    ``clip_grad_norm_`` on the way), barrier.  Replaces DDP's bucketed all-reduce (accelerator.prepare, turbo :491, sync gate
    :858) and the norm pass of ``clip_grad_norm_`` (:859).  Raises if the group has no multicast support (no NVSwitch)."""

    PARTS_PAD = 64  # floats reserved behind the gradient for the per-rank double[world] sums of squares

    def __init__(self, group=None):
        import torch.distributed as dist
        import torch.distributed._symmetric_memory as symm
        if not (dist.is_available() and dist.is_initialized()):
            raise _lib.Psob200Error("SymmetricGradExchange needs an initialised process group")
        self.group = group if group is not None else dist.group.WORLD
        self.world, self.rank = dist.get_world_size(self.group), dist.get_rank(self.group)
        if 2 * self.world > self.PARTS_PAD:
            raise _lib.Psob200Error(f"at most {self.PARTS_PAD // 2} ranks")
        self._symm = symm
        self.handle = self.buffer = None
        self.n = 0

    def allocate(self, n: int, device) -> torch.Tensor:
        """``LoRAGradBucket`` allocator: n fp32 gradient elements (+ the norm slots) in symmetric memory; collective."""
        self.n = (n + 3) // 4 * 4
        self.buffer = self._symm.empty(self.n + self.PARTS_PAD, dtype=torch.float32, device=device)
        self.buffer.zero_()
        self.handle = self._symm.rendezvous(self.buffer, self.group)
        if not getattr(self.handle, "multicast_ptr", 0):
            raise _lib.Psob200Error("this process group has no NVLink multicast mapping (multimem needs NVSwitch / NVLS)")
        torch.cuda.synchronize(device)
        self.handle.barrier(channel=0)
        return self.buffer[:n]

    @property
    def sumsq_parts_ptr(self) -> int:
        return self.buffer.data_ptr() + 4 * self.n

    def exchange(self) -> None:
        dev = self.buffer.device
        a = _lib.FlatAllreduceArgs()
        a.grad_multicast = self.handle.multicast_ptr
        a.sumsq_multicast = self.handle.multicast_ptr + 4 * self.n
        a.n, a.rank, a.world, a.scale = self.n, self.rank, self.world, 1.0 / self.world
        self.handle.barrier(channel=0)  # every rank's backward has finished accumulating into its copy
        _lib.launch(dev, "psob200_flat_allreduce_sumsq", C.byref(a), _lib.current_stream(dev))
        self.handle.barrier(channel=1)  # every slice (and every norm slot) has landed everywhere


def dynamic_quant_map(signed: bool) -> torch.Tensor:
    """bitsandbytes' ``create_dynamic_map(signed, max_exponent_bits=7, total_bits=8)``: the 256 sorted fp32 code values of
    the 8-bit optimizer state (signed for the first moment, unsigned for the second).  Decade i = 0..6 contributes the
    means of neighbouring points of ``linspace(0.1, 1, k)`` (k = 2^i + 1 signed, 2^(i+1) + 1 unsigned) times 10^(i-6), and
    their negatives when signed; then 0 and 1."""
    data = []
    for i in range(7):
        b = torch.linspace(0.1, 1, 2 ** i + 1 if signed else 2 ** (i + 1) + 1)
        means = (b[:-1] + b[1:]) / 2.0
        data += ((10 ** (i - 6)) * means).tolist()
        if signed:
            data += (-(10 ** (i - 6)) * means).tolist()
    data += [0.0, 1.0]
    return torch.tensor(sorted(data), dtype=torch.float32)


def blockwise_layout(numels, offsets, block_size: int = 256, min_8bit_size: int = 4096):
    """Block tables of the 8-bit optimizer state over a flat layout (bitsandbytes' per-tensor blocks): every matrix with
    ``numel >= min_8bit_size`` is cut into blocks of ``block_size`` elements from its own flat offset (the last one may be
    short) -> ``blocks8`` int64 [B, 2] = {flat offset, length}; smaller matrices keep fp32 moments in a compact buffer and
    are cut the same way -> ``chunks32`` int64 [C, 3] = {flat offset, length, compact offset}.  Returns
    ``(blocks8, chunks32, compact_numel)``; compact offsets are multiples of 8 like the flat ones."""
    blocks, chunks, compact = [], [], 0
    for n, off in zip(numels, offsets):
        if off % 8:
            raise ValueError(f"flat offset {off} is not a multiple of 8 elements")
        if n >= min_8bit_size:
            blocks += [(off + s, min(block_size, n - s)) for s in range(0, n, block_size)]
        else:
            chunks += [(off + s, min(block_size, n - s), compact + s) for s in range(0, n, block_size)]
            compact += (n + 7) // 8 * 8
    return (torch.tensor(blocks, dtype=torch.int64).reshape(-1, 2), torch.tensor(chunks, dtype=torch.int64).reshape(-1, 3),
            compact)


def _table_positions(table: torch.Tensor):
    """(row of each covered element, its position at column 0 + i, at column 2 + i if present) of a block / chunk table."""
    lens = table[:, 1]
    starts = torch.cumsum(lens, 0) - lens
    row = torch.repeat_interleave(torch.arange(table.shape[0], device=table.device), lens)
    i = torch.arange(int(lens.sum()), device=table.device) - starts[row]
    return row, table[row, 0] + i, (table[row, 2] + i if table.shape[1] > 2 else None)


class FusedLoRAOptimizer:
    """The optimizer boundary of the training step on the flat LoRA buffers: ``clip_grad_norm_`` + AdamW +
    ``zero_grad`` + refresh of the 16-bit GEMM operands in two kernel launches (psob200_flat_adamw_step) instead of the
    reference's per-parameter kernels (train_online_pso_sdxl_turbo.py:428-448 optimizer, :859 clipping, :860-861
    step / zero_grad).  Parameters, gradients and both Adam moments of every adapter matrix are slices of four flat
    fp32 buffers with one layout; ``self.bucket`` is the gradient buffer (``all_reduce()`` = the data-parallel exchange).
    Update rule = ``torch.optim.AdamW`` (decoupled weight decay, bias correction).

    ``optim_bits=8`` is the Turbo recipe's ``use_8bit_adam`` (bitsandbytes ``AdamW(optim_bits=8)``, same keyword names):
    blockwise 8-bit moments (``block_size`` elements per fp32 absmax; matrices below ``min_8bit_size`` elements keep fp32
    moments), bitsandbytes' update rule (weight decay after the step), one update launch of psob200_flat_adamw8_step.
    ``exp_avg`` / ``exp_avg_sq`` are then None; ``dequantized_moments()`` gives flat fp32 copies.

    ``grad_scaler`` (an ``amp.DeviceGradScaler``, fp16 training: GradScaler around :857-860): the boundary unscales by
    ``1 / S`` read on the device (times ``grad_scale``), skips the update on a non-finite norm and updates ``S`` and the
    growth tracker in the same launch -- ``step()`` stays free of host syncs and capturable in a CUDA graph."""

    def __init__(self, model: nn.Module, lr: float = 1e-5, betas=(0.9, 0.999), eps: float = 1e-8,
                 weight_decay: float = 1e-4, max_grad_norm: float = 1.0, exchange: Optional[SymmetricGradExchange] = None,
                 optim_bits: int = 32, block_size: int = 256, min_8bit_size: int = 4096, grad_scaler=None):
        if optim_bits not in (8, 32):
            raise ValueError(f"optim_bits must be 8 or 32, got {optim_bits}")
        if optim_bits == 8 and block_size not in (256, 2048):
            raise ValueError(f"block_size must be 256 or 2048, got {block_size}")
        self.optim_bits, self.block_size, self.min_8bit_size = optim_bits, block_size, min_8bit_size
        self.exchange = exchange  # None: all_reduce() is one NCCL call; else the fused NVLink-multicast kernel
        self.layers = lora_layers(model)
        self.groups = projection_groups(model)
        params = lora_parameters(model)
        if any(p.dtype != torch.float32 for p in params):
            raise _lib.Psob200Error("FusedLoRAOptimizer trains fp32 adapter parameters (the shipped mixed-precision recipes)")
        _lib.require_cuda(*params)
        self.bucket = LoRAGradBucket(params, align=8, allocator=exchange.allocate if exchange is not None else None)
        self._parts_ready = False
        flat = self.bucket.flat
        self.flat_param = torch.zeros_like(flat)
        # what state_dict() carries: the state tensors (attribute names) and the keys that describe their format
        if optim_bits == 32:
            self._state_names, self._format = ("flat_param", "exp_avg", "exp_avg_sq"), {}
            self.exp_avg = torch.zeros_like(flat)
            self.exp_avg_sq = torch.zeros_like(flat)
        else:
            self._state_names = ("flat_param", "code1", "code2", "absmax1", "absmax2", "exp_avg32", "exp_avg_sq32", "qmap1",
                                 "qmap2")
            self._format = {"optim_bits": 8, "block_size": block_size, "min_8bit_size": min_8bit_size}
            self.exp_avg = self.exp_avg_sq = None
            blocks8, chunks32, n32 = blockwise_layout([p.numel() for p in self.bucket.params], self.bucket.offsets,
                                                      block_size, min_8bit_size)
            dev = flat.device
            self.blocks8, self.chunks32 = blocks8.to(dev), chunks32.to(dev)
            self.qmap1, self.qmap2 = dynamic_quant_map(True).to(dev), dynamic_quant_map(False).to(dev)
            self.code1 = torch.full((flat.numel(),), 127, dtype=torch.uint8, device=dev)  # qmap1[127] == 0
            self.code2 = torch.zeros(flat.numel(), dtype=torch.uint8, device=dev)         # qmap2[0] == 0
            self.absmax1 = torch.zeros(blocks8.shape[0], dtype=torch.float32, device=dev)
            self.absmax2 = torch.zeros_like(self.absmax1)
            self.exp_avg32 = torch.zeros(n32, dtype=torch.float32, device=dev)
            self.exp_avg_sq32 = torch.zeros_like(self.exp_avg32)
        op_dtype = self.layers[0].base_layer.weight.dtype
        self.flat_operand = torch.zeros(flat.numel(), dtype=op_dtype, device=flat.device)
        self.workspace = torch.zeros(2, dtype=torch.float64, device=flat.device)
        self.grad_norm = torch.zeros(1, dtype=torch.float32, device=flat.device)
        # fp16 loss scaling (accelerate's GradScaler, turbo :126 / :857-860): `grad_scale` is the unscale factor of the next
        # step(); a non-finite norm skips the update on the device, sets `found_inf` and does not advance `step_dev`
        self.found_inf = torch.zeros(1, dtype=torch.float32, device=flat.device)
        self.step_dev = torch.zeros(1, dtype=torch.int64, device=flat.device)  # applied updates (bias correction)
        self.grad_scale = 1.0
        self.grad_scaler = grad_scaler
        if grad_scaler is not None:
            amp.scaler_arg(grad_scaler, flat.device)  # a DeviceGradScaler on this device, or raise now
        self.lr, self.betas, self.eps, self.weight_decay, self.max_grad_norm = lr, betas, eps, weight_decay, max_grad_norm
        self.step_count = 0  # step() calls (host side, no sync); applied updates are counted in `step_dev`
        self._unbacked = []  # adapter matrices whose operand copy needs a padded pitch (rank not a multiple of 8)
        by_param = {}
        for lay in self.layers:
            n = lay.active_adapter
            by_param[id(lay.lora_A[n].weight)] = (lay, "a")
            by_param[id(lay.lora_B[n].weight)] = (lay, "b")
        for p, off in zip(self.bucket.params, self.bucket.offsets):
            view = self.flat_param[off:off + p.numel()].view(p.shape)
            view.copy_(p.detach())
            p.data = view  # the parameter now lives in the flat buffer
            lay, which = by_param[id(p)]
            if p.shape[1] % 8 == 0:
                op = self.flat_operand[off:off + p.numel()].view(p.shape)
                op.copy_(view)
                lay.install_operand(which, op_dtype, op)  # kept current by the fused kernel
            else:
                self._unbacked.append((lay, which, op_dtype))

    def all_reduce(self, group=None):
        """The data-parallel exchange: mean of the flat gradient over the ranks.  With a ``SymmetricGradExchange`` it is
        one launch of ours (which also leaves the norm of the averaged gradient for ``step()``), else one NCCL call."""
        if self.exchange is not None:
            self.exchange.exchange()
            self._parts_ready = True
            return None
        return self.bucket.all_reduce(group)

    def step(self) -> torch.Tensor:
        """Clip, update, zero the gradient, refresh the operands.  Returns the (pre-clip) gradient norm, on the device."""
        self.step_count += 1
        entry, a, extra = self._launch_args()
        if self._parts_ready:  # the fused exchange already produced the sum of squares, one piece per rank
            a.n_sumsq_parts, a.sumsq_parts = self.exchange.world, self.exchange.sumsq_parts_ptr
            self._parts_ready = False
        _lib.launch(self.flat_param.device, entry, C.byref(a), *extra, _lib.current_stream(self.flat_param.device))
        self._refresh_unbacked()
        return self.grad_norm

    def _launch_args(self):
        """``(entry point, argument struct, further arguments)`` of this optimizer's boundary for the next ``step()`` (norm
        computed in-launch); the call is ``entry(byref(struct), *further, stream)``.  With a loss scaler the entry point is
        the ``_scaled`` one and ``further`` holds the scaler."""
        extra = ()
        if self.optim_bits == 32:
            entry, a = "psob200_flat_adamw_step", _lib.FlatAdamwArgs()
            a.exp_avg, a.exp_avg_sq = self.exp_avg.data_ptr(), self.exp_avg_sq.data_ptr()
        else:
            entry, a = "psob200_flat_adamw8_step", _lib.FlatAdamw8Args()
            a.code1, a.code2 = self.code1.data_ptr(), self.code2.data_ptr()
            a.absmax1, a.absmax2 = self.absmax1.data_ptr(), self.absmax2.data_ptr()
            a.map1, a.map2 = self.qmap1.data_ptr(), self.qmap2.data_ptr()
            a.blocks8, a.n_blocks8 = self.blocks8.data_ptr(), self.blocks8.shape[0]
            a.chunks32, a.n_chunks32 = self.chunks32.data_ptr(), self.chunks32.shape[0]
            a.exp_avg32, a.exp_avg_sq32 = self.exp_avg32.data_ptr(), self.exp_avg_sq32.data_ptr()
            a.block_size = self.block_size
        a.param, a.grad = self.flat_param.data_ptr(), self.bucket.flat.data_ptr()
        a.operand, a.operand_dtype = self.flat_operand.data_ptr(), _lib.dtype_code(self.flat_operand)
        a.norm_out, a.workspace = self.grad_norm.data_ptr(), self.workspace.data_ptr()
        a.n, a.step = self.flat_param.numel(), self.step_count
        a.lr, a.beta1, a.beta2, a.eps = self.lr, self.betas[0], self.betas[1], self.eps
        a.weight_decay, a.max_grad_norm, a.grad_scale = self.weight_decay, self.max_grad_norm, float(self.grad_scale)
        a.found_inf, a.step_dev = self.found_inf.data_ptr(), self.step_dev.data_ptr()
        if self.grad_scaler is not None:
            entry, extra = entry + "_scaled", (C.byref(amp.scaler_arg(self.grad_scaler, self.flat_param.device)),)
        return entry, a, extra

    def dequantized_moments(self) -> tuple[torch.Tensor, torch.Tensor]:
        """Flat fp32 copies of both Adam moments in the parameter layout (8-bit blocks dequantised as the kernel does:
        ``qmap[code] * absmax``), for inspection and tests.  Elements outside every matrix are 0."""
        if self.optim_bits == 32:
            return self.exp_avg.clone(), self.exp_avg_sq.clone()
        m = torch.zeros_like(self.flat_param)
        v = torch.zeros_like(self.flat_param)
        if self.blocks8.shape[0]:
            blk, pos, _ = _table_positions(self.blocks8)
            m[pos] = self.qmap1[self.code1[pos].long()] * self.absmax1[blk]
            v[pos] = self.qmap2[self.code2[pos].long()] * self.absmax2[blk]
        if self.chunks32.shape[0]:
            _, pos, cpos = _table_positions(self.chunks32)
            m[pos], v[pos] = self.exp_avg32[cpos], self.exp_avg_sq32[cpos]
        return m, v

    def _refresh_unbacked(self) -> None:
        for lay, which, dt in self._unbacked:  # padded-pitch copies: re-made in place by the layer itself
            lay.refresh_operand(which, dt)
        for g in self.groups:  # stacked groups that keep private (padded) operand copies: re-stacked in place
            g.refresh_private_operands()

    def zero_grad(self, set_to_none: bool = False) -> None:
        """In-place zero of the flat gradient (``step()`` already leaves it zeroed); ``param.grad`` stays a bucket view."""
        self.bucket.zero_grad(set_to_none)

    # ---- checkpoint / resume (accelerator.save_state / load_state, turbo :889: the AdamW moments and step count travel too)
    def state_dict(self) -> dict:
        """Everything a resumed run needs for bit-identical continuation: the fp32 master parameters, both Adam moments,
        the count of applied updates (one host sync) and the hyper-parameters.  Tensors are clones on the optimizer's device.
        With ``optim_bits=8`` the moments are the 8-bit state instead (codes, absmax, compact fp32 moments, both maps) and
        the dict also records ``optim_bits``, ``block_size`` and ``min_8bit_size``.  With a loss scaler attached it also
        holds ``scaler_scale`` / ``scaler_growth_tracker`` (the device state) and ``scaler`` (its hyper-parameters)."""
        sd = {k: getattr(self, k).clone() for k in self._state_names}
        if self.grad_scaler is not None:
            s = self.grad_scaler
            sd["scaler_scale"], sd["scaler_growth_tracker"] = s.scale_tensor.clone(), s.growth_tracker.clone()
            sd["scaler"] = s.hyper()
        sd.update({"step": int(self.step_dev.item()), "step_calls": int(self.step_count),
                   "hyper": {"lr": self.lr, "beta1": self.betas[0], "beta2": self.betas[1], "eps": self.eps,
                             "weight_decay": self.weight_decay, "max_grad_norm": self.max_grad_norm},
                   "layout": {"numel": int(self.flat_param.numel()), "offsets": [int(o) for o in self.bucket.offsets],
                              "shapes": [list(p.shape) for p in self.bucket.params]}})
        sd.update(self._format)
        return sd

    def load_state_dict(self, sd: dict, load_hyper: bool = True) -> None:
        """Inverse of ``state_dict()``.  The parameters live in ``flat_param`` (every adapter ``weight`` is a view of it), so
        loading also restores the adapters; the 16-bit operand copies the GEMM kernels read are refreshed; the gradient is zeroed.
        Loss-scaler state loads into the attached scaler (one without such state in ``sd`` keeps its values, as a fresh fp16
        run would); scaler state with no scaler attached is refused rather than dropped."""
        has_scaler_state = "scaler_scale" in sd
        if has_scaler_state and self.grad_scaler is None:
            raise _lib.Psob200Error("the optimizer state holds loss-scaler state (an fp16 run) but this optimizer has no "
                                    "grad_scaler: pass grad_scaler=DeviceGradScaler(...) so that it is restored, not dropped")
        bits = int(sd.get("optim_bits", 32))  # fp32 state records no format keys
        if bits != self.optim_bits:
            raise _lib.Psob200Error(f"optimizer state was saved with optim_bits={bits}; this optimizer has optim_bits="
                                    f"{self.optim_bits} (the moments of the two modes are stored differently)")
        if any(int(sd[k]) != v for k, v in self._format.items()):
            raise _lib.Psob200Error("8-bit optimizer state was saved with " + ", ".join(f"{k}={sd[k]}" for k in self._format)
                                    + "; this optimizer has " + ", ".join(f"{k}={v}" for k, v in self._format.items()))
        lay = sd["layout"]
        if lay["numel"] != self.flat_param.numel() or list(lay["offsets"]) != [int(o) for o in self.bucket.offsets] or \
                [list(x) for x in lay["shapes"]] != [list(p.shape) for p in self.bucket.params]:
            raise _lib.Psob200Error("optimizer state was saved for a different flat layout: rank / target modules differ, or "
                                    "fuse_attention_projections / fuse_cross_attention_kv were not called the same way before "
                                    "the optimizer was built (lora_parameters() orders the buffers by group and bank)")
        dev = self.flat_param.device
        if bits == 8 and not (torch.equal(sd["qmap1"].cpu(), self.qmap1.cpu()) and torch.equal(sd["qmap2"].cpu(), self.qmap2.cpu())):
            raise _lib.Psob200Error("8-bit optimizer state was saved with other quantisation maps")
        with torch.no_grad():
            for k in self._state_names:
                getattr(self, k).copy_(sd[k].to(dev))
            self.step_dev.fill_(int(sd["step"]))
            self.flat_operand.copy_(self.flat_param)  # what psob200_flat_adamw_step would have left
            if has_scaler_state:
                s = self.grad_scaler
                s.set_hyper(**sd["scaler"])
                s.scale_tensor.copy_(sd["scaler_scale"].to(device=s.device, dtype=torch.float32).reshape(1))
                s.growth_tracker.copy_(sd["scaler_growth_tracker"].to(device=s.device, dtype=torch.int32).reshape(1))
        self.step_count = int(sd.get("step_calls", sd["step"]))
        if load_hyper:
            h = sd["hyper"]
            self.lr, self.betas, self.eps = h["lr"], (h["beta1"], h["beta2"]), h["eps"]
            self.weight_decay, self.max_grad_norm = h["weight_decay"], h["max_grad_norm"]
        self._refresh_unbacked()
        self.bucket.zero_grad()
        self._parts_ready = False


# ----------------------------------------------------------------------------------------------- attention processor
class PSOAttnProcessor2_0:
    """diffusers==0.27.0 ``AttnProcessor2_0``: same ``__call__`` signature, same data flow; the four projections run
    on the tcgen05 path when they are ``LoRALinear`` (the attention core stays ``F.scaled_dot_product_attention``,
    which is outside the PSO hot path)."""

    def __call__(self, attn, hidden_states, encoder_hidden_states=None, attention_mask=None, temb=None, scale=1.0):
        residual = hidden_states
        if getattr(attn, "spatial_norm", None) is not None:
            hidden_states = attn.spatial_norm(hidden_states, temb)
        input_ndim = hidden_states.ndim
        if input_ndim == 4:
            bsz, ch, h, w = hidden_states.shape
            hidden_states = hidden_states.view(bsz, ch, h * w).transpose(1, 2)
        bsz = hidden_states.shape[0]
        if getattr(attn, "group_norm", None) is not None:
            hidden_states = attn.group_norm(hidden_states.transpose(1, 2)).transpose(1, 2)
        groups = attn.__dict__.get("_psob200_groups")  # lora.fuse_attention_projections: stacked q / k / v (or k / v) launches
        if encoder_hidden_states is None and groups is not None and "qkv" in groups:
            query, key, value = groups["qkv"](hidden_states)
        else:
            query = attn.to_q(hidden_states)
            if encoder_hidden_states is None:
                encoder_hidden_states = hidden_states
            elif getattr(attn, "norm_cross", None):
                encoder_hidden_states = attn.norm_encoder_hidden_states(encoder_hidden_states)
            # fuse_cross_attention_kv: produced by the bank launch at the start of this forward.  Not popped: a gradient-checkpointed
            # block runs again in the backward and must take the same path (the bank's next launch overwrites the entry)
            pre = attn.__dict__.get("_psob200_kv")
            if pre is not None and not (pre[3]["live"] or torch._C._current_graph_task_id() != -1):
                pre = None  # left over from an earlier forward: only that forward and its backward may use it
            if pre is not None and pre[0] is encoder_hidden_states:
                key, value = pre[1], pre[2]
            elif groups is not None and "kv" in groups:
                key, value = groups["kv"](encoder_hidden_states)
            else:
                key = attn.to_k(encoder_hidden_states)
                value = attn.to_v(encoder_hidden_states)
        inner = key.shape[-1]
        hd = inner // attn.heads
        query = query.view(bsz, -1, attn.heads, hd).transpose(1, 2)
        key = key.view(bsz, -1, attn.heads, hd).transpose(1, 2)
        value = value.view(bsz, -1, attn.heads, hd).transpose(1, 2)
        if attention_mask is not None and hasattr(attn, "prepare_attention_mask"):
            attention_mask = attn.prepare_attention_mask(attention_mask, key.shape[2], bsz)
            attention_mask = attention_mask.view(bsz, attn.heads, -1, attention_mask.shape[-1])
        hidden_states = F.scaled_dot_product_attention(query, key, value, attn_mask=attention_mask, dropout_p=0.0,
                                                       is_causal=False)
        hidden_states = hidden_states.transpose(1, 2).reshape(bsz, -1, attn.heads * hd).to(query.dtype)
        hidden_states = attn.to_out[0](hidden_states)
        hidden_states = attn.to_out[1](hidden_states)
        if input_ndim == 4:
            hidden_states = hidden_states.transpose(-1, -2).reshape(bsz, ch, h, w)
        if getattr(attn, "residual_connection", False):
            hidden_states = hidden_states + residual
        rescale = getattr(attn, "rescale_output_factor", 1.0)
        return hidden_states if rescale == 1.0 else hidden_states / rescale  # x / 1.0 would still launch a kernel

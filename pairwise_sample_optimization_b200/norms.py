"""LayerNorm and GroupNorm of the UNet on fused kernels, forward and backward (psob200_layer_norm_* / psob200_group_norm_*).

Replaces ``torch.nn.LayerNorm`` (one normalised dimension), ``torch.nn.GroupNorm``, and in diffusers==0.27.0
``ResnetBlock2D.forward`` the lines::

    hidden_states = self.nonlinearity(self.norm1(input_tensor))
    hidden_states = self.norm2(hidden_states + self.time_emb_proj(self.nonlinearity(temb))[:, :, None, None])
    hidden_states = self.nonlinearity(hidden_states)

with one GroupNorm kernel pair each (SiLU and the time-embedding add fused).  Not rows of the PSO hot path (SURVEY.md
section 8): the stock norm and SiLU kernels were 15 % of the measured micro-step's kernel time.  The autograd functions
save the input (and the time-embedding term) plus fp32 mean / rstd per row or group, never the normalised output.
The base UNet is frozen, so the kernels compute no weight, bias or time-embedding gradient: ``layer_norm`` / ``group_norm``
raise when one would be needed, and the forwards ``install_fused_norms`` patches in take the stock path then.
No PyTorch fallback otherwise: CPU tensors raise.
"""
from __future__ import annotations

import ctypes as C

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import _lib

_LN_MAX_C = 2048  # psob200_layer_norm_*: C a multiple of 8, at most 2048


def _out_dtype(x: torch.Tensor) -> torch.dtype:
    """What the stock op returns: fp32 for 16-bit input under an active CUDA autocast (layer_norm and group_norm are on
    autocast's fp32 list), else the input's type.  The kernels read the 16-bit input directly: no cast kernel."""
    if x.dtype in (torch.bfloat16, torch.float16) and torch.is_autocast_enabled("cuda"):
        return torch.float32
    return x.dtype


def _empty(shape, dtype, device) -> torch.Tensor:
    """torch.empty without the NaN fill that deterministic mode adds: the kernels write every element of what this returns."""
    det = torch.utils.deterministic
    if not (det.fill_uninitialized_memory and torch.are_deterministic_algorithms_enabled()):
        return torch.empty(shape, dtype=dtype, device=device)
    det.fill_uninitialized_memory = False
    try:
        return torch.empty(shape, dtype=dtype, device=device)
    finally:
        det.fill_uninitialized_memory = True


def _affine(weight, bias):
    """(weight ptr, bias ptr, dtype code) of the optional affine parameters (fp32 code when both are absent)."""
    if weight is not None and bias is not None and weight.dtype != bias.dtype:
        raise _lib.Psob200Error(f"weight and bias must share a dtype, got {weight.dtype} and {bias.dtype}")
    for t in (weight, bias):
        if t is not None and not t.is_contiguous():
            raise _lib.Psob200Error("weight and bias must be contiguous")
    p = weight if weight is not None else bias
    ptr = lambda t: t.data_ptr() if t is not None else None
    return ptr(weight), ptr(bias), (_lib.dtype_code(p) if p is not None else _lib.F32)


def _check_no_grad_needed(*tensors) -> None:
    if torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in tensors):
        raise _lib.Psob200Error("the fused norms compute no weight / bias / channel_add gradient (the base model is frozen); "
                                "use the stock op for trainable affine parameters")


class _LayerNormFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias, eps, out_dtype):
        dev = _lib.require_cuda(x, weight, bias)
        width = x.shape[-1]
        x2 = x.detach().contiguous().view(-1, width)
        rows = x2.shape[0]
        y = _empty((rows, width), out_dtype, dev)
        mean, rstd = _empty((rows,), torch.float32, dev), _empty((rows,), torch.float32, dev)
        a = _lib.LayerNormArgs()
        a.weight, a.bias, a.param_dtype = _affine(weight, bias)
        a.x, a.y, a.mean, a.rstd = x2.data_ptr(), y.data_ptr(), mean.data_ptr(), rstd.data_ptr()
        a.rows, a.C, a.ld_x, a.ld_y, a.eps = rows, width, width, width, eps
        a.dtype, a.out_dtype = _lib.dtype_code(x2), _lib.dtype_code(y)
        _lib.launch(dev, "psob200_layer_norm_forward", C.byref(a), _lib.current_stream(dev))
        ctx.save_for_backward(x2, weight, bias, mean, rstd)
        ctx.shape, ctx.out_dtype = x.shape, out_dtype
        return y.view(x.shape)

    @staticmethod
    def backward(ctx, dy):
        x2, weight, bias, mean, rstd = ctx.saved_tensors
        rows, width = x2.shape
        d2 = dy.reshape(rows, width).to(ctx.out_dtype).contiguous()
        dx = _empty((rows, width), x2.dtype, x2.device)
        a = _lib.LayerNormArgs()
        a.weight, a.bias, a.param_dtype = _affine(weight, bias)
        a.x, a.dy, a.dx, a.mean, a.rstd = x2.data_ptr(), d2.data_ptr(), dx.data_ptr(), mean.data_ptr(), rstd.data_ptr()
        a.rows, a.C, a.ld_x, a.ld_dy, a.ld_dx = rows, width, width, width, width
        a.dtype, a.out_dtype = _lib.dtype_code(x2), _lib.dtype_code(d2)
        _lib.launch(x2.device, "psob200_layer_norm_backward", C.byref(a), _lib.current_stream(x2.device))
        return dx.view(ctx.shape), None, None, None, None


class _GroupNormFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, channel_add, weight, bias, num_groups, eps, silu, out_dtype):
        dev = _lib.require_cuda(x, channel_add, weight, bias)
        if x.dim() < 2:
            raise _lib.Psob200Error(f"group_norm needs an [N, C, *] input, got shape {tuple(x.shape)}")
        n, c = x.shape[0], x.shape[1]
        x2 = x.detach().contiguous()
        ca = None
        if channel_add is not None:
            if channel_add.dtype != x.dtype or channel_add.numel() != n * c:
                raise _lib.Psob200Error(f"channel_add must be [N, C] = [{n}, {c}] of {x.dtype}, got "
                                        f"{tuple(channel_add.shape)} of {channel_add.dtype}")
            ca = channel_add.detach().reshape(n, c).contiguous()
        y = _empty(x2.shape, out_dtype, dev)
        mean, rstd = _empty((n * num_groups,), torch.float32, dev), _empty((n * num_groups,), torch.float32, dev)
        a, _ws = _GroupNormFn._args(x2, ca, weight, bias, num_groups, eps, silu, mean, rstd, dev)
        a.y, a.out_dtype = y.data_ptr(), _lib.dtype_code(y)
        _lib.launch(dev, "psob200_group_norm_forward", C.byref(a), _lib.current_stream(dev))
        ctx.save_for_backward(x2, ca, weight, bias, mean, rstd)
        ctx.num_groups, ctx.eps, ctx.silu, ctx.out_dtype = num_groups, eps, silu, out_dtype
        return y

    @staticmethod
    def backward(ctx, dy):
        x2, ca, weight, bias, mean, rstd = ctx.saved_tensors
        d2 = dy.to(ctx.out_dtype).contiguous()
        dx = _empty(x2.shape, x2.dtype, x2.device)
        a, _ws = _GroupNormFn._args(x2, ca, weight, bias, ctx.num_groups, ctx.eps, ctx.silu, mean, rstd, x2.device)
        a.dy, a.dx, a.out_dtype = d2.data_ptr(), dx.data_ptr(), _lib.dtype_code(d2)
        _lib.launch(x2.device, "psob200_group_norm_backward", C.byref(a), _lib.current_stream(x2.device))
        return dx, None, None, None, None, None, None, None

    @staticmethod
    def _args(x2, ca, weight, bias, num_groups, eps, silu, mean, rstd, dev):
        n, c = x2.shape[0], x2.shape[1]
        hw = x2.numel() // (n * c)
        ws_bytes = _lib.lib().psob200_group_norm_workspace_bytes(n, c, hw, num_groups)
        ws = _empty((max(ws_bytes, 16),), torch.uint8, dev)  # cross-CTA partials of this call; no initialisation needed
        a = _lib.GroupNormArgs()
        a.weight, a.bias, a.param_dtype = _affine(weight, bias)
        a.x, a.channel_add, a.mean, a.rstd = x2.data_ptr(), (ca.data_ptr() if ca is not None else None), mean.data_ptr(), rstd.data_ptr()
        a.workspace, a.workspace_bytes = ws.data_ptr(), ws.numel()
        a.N, a.C, a.HW, a.G, a.eps, a.silu = n, c, hw, num_groups, eps, int(silu)
        a.dtype = _lib.dtype_code(x2)
        return a, ws  # the caller holds the workspace until the launch is enqueued


def layer_norm(x: torch.Tensor, weight: torch.Tensor | None = None, bias: torch.Tensor | None = None,
               eps: float = 1e-5) -> torch.Tensor:
    """``F.layer_norm(x, (x.shape[-1],), weight, bias, eps)`` on the fused kernels, differentiable in ``x``."""
    _check_no_grad_needed(weight, bias)
    return _LayerNormFn.apply(x, weight, bias, float(eps), _out_dtype(x))


def group_norm(x: torch.Tensor, num_groups: int, weight: torch.Tensor | None = None, bias: torch.Tensor | None = None,
               eps: float = 1e-5, *, silu: bool = False, channel_add: torch.Tensor | None = None) -> torch.Tensor:
    """``F.group_norm(x + channel_add[:, :, None, None], num_groups, weight, bias, eps)`` followed by ``F.silu`` when
    ``silu``, on the fused kernels, differentiable in ``x``.  ``channel_add`` ([N, C], x's dtype) is added and rounded to
    x's dtype first, as the stock add does."""
    _check_no_grad_needed(weight, bias, channel_add)
    return _GroupNormFn.apply(x, channel_add, weight, bias, int(num_groups), float(eps), bool(silu), _out_dtype(x))


# ------------------------------------------------------------------------------------------------------------ module patches
def _grad_needed(*tensors) -> bool:
    return torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in tensors)


def _is_resnet_block(m: nn.Module) -> bool:
    """diffusers' ResnetBlock2D (or a module of that name and surface) whose forward is the three lines above."""
    if type(m).__name__ != "ResnetBlock2D":
        return False
    if not all(hasattr(m, k) for k in ("norm1", "conv1", "time_emb_proj", "norm2", "conv2", "conv_shortcut")):
        return False
    if not (isinstance(m.norm1, nn.GroupNorm) and isinstance(m.norm2, nn.GroupNorm)):
        return False
    if hasattr(m, "time_embedding_norm"):  # diffusers' class: only its default configuration has that data flow
        return (m.time_embedding_norm == "default" and getattr(m, "upsample", None) is None
                and getattr(m, "downsample", None) is None and getattr(m, "output_scale_factor", 1.0) == 1.0
                and not getattr(m, "skip_time_act", False) and getattr(getattr(m, "dropout", None), "p", 0.0) == 0.0
                and isinstance(getattr(m, "nonlinearity", None), nn.SiLU))
    return True


def _layer_norm_forward(m: nn.LayerNorm):
    stock = type(m).forward.__get__(m)

    def forward(x):
        if _grad_needed(m.weight, m.bias):
            return stock(x)
        return layer_norm(x, m.weight, m.bias, m.eps)
    return forward


def _group_norm_forward(m: nn.GroupNorm):
    stock = type(m).forward.__get__(m)

    def forward(x):
        if _grad_needed(m.weight, m.bias):
            return stock(x)
        return group_norm(x, m.num_groups, m.weight, m.bias, m.eps)
    return forward


def _resnet_forward(m: nn.Module):
    stock = type(m).forward.__get__(m)

    def forward(x, temb, *args, **kwargs):
        n1, n2 = m.norm1, m.norm2
        if args or kwargs or _grad_needed(n1.weight, n1.bias, n2.weight, n2.bias, temb):
            return stock(x, temb, *args, **kwargs)
        h = m.conv1(group_norm(x, n1.num_groups, n1.weight, n1.bias, n1.eps, silu=True))
        t = None
        if m.time_emb_proj is not None and temb is not None:
            t = m.time_emb_proj(F.silu(temb))
            if t.dtype != h.dtype:  # the kernel adds a term of x's own type; the stock add promotes
                h, t = h + t[:, :, None, None], None
        h = m.conv2(group_norm(h, n2.num_groups, n2.weight, n2.bias, n2.eps, silu=True, channel_add=t))
        return (x if m.conv_shortcut is None else m.conv_shortcut(x)) + h
    return forward


def install_fused_norms(model: nn.Module) -> dict:
    """Point the norms of ``model`` at the fused kernels (opt-in, like ``feed_forward.install_fused_geglu``):

    * every ``nn.LayerNorm`` over one dimension whose width the kernel takes (a multiple of 8, at most 2048);
    * every ``nn.GroupNorm``;
    * every ResnetBlock2D-shaped module (``_is_resnet_block``): ``norm1`` + SiLU and time-embedding add + ``norm2`` + SiLU
      on one GroupNorm kernel pair each.

    A patched forward takes the stock path when a norm weight or bias, or the block's ``temb``, requires grad (the kernels
    compute no such gradient), so installing never changes which gradients exist.  Returns the number of modules patched
    per kind: ``{"layer_norm": .., "group_norm": .., "resnet_block": ..}``."""
    counts = {"layer_norm": 0, "group_norm": 0, "resnet_block": 0}
    for m in model.modules():
        if isinstance(m, nn.LayerNorm) and len(m.normalized_shape) == 1 and m.normalized_shape[0] % 8 == 0 \
                and m.normalized_shape[0] <= _LN_MAX_C:
            m.forward = _layer_norm_forward(m)
            counts["layer_norm"] += 1
        elif isinstance(m, nn.GroupNorm):
            m.forward = _group_norm_forward(m)
            counts["group_norm"] += 1
        elif _is_resnet_block(m):
            m.forward = _resnet_forward(m)
            counts["resnet_block"] += 1
    return counts

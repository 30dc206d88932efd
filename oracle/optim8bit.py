"""Blockwise 8-bit AdamW (bitsandbytes ``AdamW(optim_bits=8)``; Dettmers et al. 2022, "8-bit Optimizers via Block-wise
Quantization") over the flat LoRA layout -- the optimizer of the Turbo recipe's ``use_8bit_adam`` (turbo T:428-448).

Parity status: restated, unpinned against the package.  bitsandbytes is third-party and absent here; this follows its
published ``create_dynamic_map`` and blockwise 8-bit Adam kernel as described in the library's documentation and paper:

* maps: ``create_dynamic_map(signed, max_exponent_bits=7, total_bits=8)`` -- signed for the first moment, unsigned for
  the second;
* blocks are per tensor: a matrix with ``numel >= min_8bit_size`` is cut into ``block_size`` blocks from its own start
  (the last may be short), one fp32 absmax per block and moment; smaller matrices keep fp32 moments;
* per element, fp32, every operation rounded on its own:
  ``m = map1[c1] absmax1; v = map2[c2] absmax2; m = m b1 + (1 - b1) g; v = v b2 + (1 - b2) g g;
  p = p + ((-lr bc2) / bc1) (m / (sqrt(v) + eps bc2)); p = p (1 - lr wd)`` (decay AFTER the step, torch decays before),
  ``bc1 = 1 - b1^t``, ``bc2 = sqrt(1 - b2^t)``;
* new absmax = max |m| (|v|) of the block; code = number of the 255 midpoints of neighbouring map entries strictly below
  ``m / absmax``; first moment only: when the chosen entry's sign bit differs from m's, step one code towards m's side.

The clip coefficient, ``grad_scale`` and the overflow skip are those of ``lora.FusedLoRAOptimizer`` (torch / accelerate).
"""
from __future__ import annotations

import math

import numpy as np
import torch

f32 = np.float32


def create_dynamic_map(signed: bool = True, max_exponent_bits: int = 7, total_bits: int = 8) -> np.ndarray:
    data = []
    non_sign_bits = total_bits - 1
    for i in range(max_exponent_bits):
        k = (2 ** (i + non_sign_bits - max_exponent_bits) + 1 if signed
             else 2 ** (i + non_sign_bits - max_exponent_bits + 1) + 1)
        boundaries = torch.linspace(0.1, 1, k)
        means = (boundaries[:-1] + boundaries[1:]) / 2.0
        data += ((10 ** (-(max_exponent_bits - 1) + i)) * means).tolist()
        if signed:
            data += (-(10 ** (-(max_exponent_bits - 1) + i)) * means).tolist()
    data.append(0)
    data.append(1.0)
    assert len(data) == 2 ** total_bits
    data.sort()
    return torch.tensor(data, dtype=torch.float32).numpy()


def midpoints(qmap: np.ndarray) -> np.ndarray:
    return (qmap[:-1] + qmap[1:]) * f32(0.5)


def quantize(x: np.ndarray, qmap: np.ndarray, m: np.ndarray | None = None) -> np.ndarray:
    """Codes of normalised values ``x``; with ``m`` (the first moment) the sign rule is applied."""
    c = np.searchsorted(midpoints(qmap), x, side="left").astype(np.int64)
    if m is not None:
        flip = np.signbit(qmap[c]) != np.signbit(m)
        c = np.where(flip, np.where(m > 0, c + 1, c - 1), c)
    return c.astype(np.uint8)


def table_positions(table: np.ndarray):
    """(row of each covered element, flat position, compact position or None) of a block / chunk table."""
    lens = table[:, 1].astype(np.int64)
    starts = np.cumsum(lens) - lens
    row = np.repeat(np.arange(table.shape[0]), lens)
    i = np.arange(int(lens.sum())) - starts[row]
    return row, table[row, 0] + i, (table[row, 2] + i if table.shape[1] > 2 else None)


def clip_coef(norm: float, max_grad_norm: float, grad_scale: float) -> np.float32:
    """``flat_adamw_kernel``'s coefficient, from the (already grad_scale-multiplied) fp32 norm."""
    if max_grad_norm > 0:
        return f32(min(f32(1.0), f32(max_grad_norm) / (f32(norm) + f32(1e-6)))) * f32(grad_scale)
    return f32(grad_scale)


def adamw8_step(state: dict, p: np.ndarray, g: np.ndarray, blocks8: np.ndarray, chunks32: np.ndarray, norm: float, t: int,
                lr: float, beta1: float, beta2: float, eps: float, weight_decay: float, max_grad_norm: float,
                grad_scale: float = 1.0):
    """One boundary.  ``state``: code1 / code2 (uint8, flat positions), absmax1 / absmax2 (per block), exp_avg32 /
    exp_avg_sq32 (compact), qmap1 / qmap2.  ``t``: 1-based count of applied updates.  Returns (p, new state); a
    non-finite ``norm`` returns both unchanged (the caller zeroes the gradient either way)."""
    p, st = p.copy(), {k: v.copy() for k, v in state.items()}
    if not math.isfinite(norm):
        return p, st
    coef = clip_coef(norm, max_grad_norm, grad_scale)
    b1, b2 = f32(beta1), f32(beta2)
    bc1 = f32(1.0 - float(b1) ** t)
    bc2 = f32(math.sqrt(1.0 - float(b2) ** t))
    step_size = (f32(-lr) * bc2) / bc1
    eps_bc2 = f32(eps) * bc2
    omb1, omb2 = f32(1) - b1, f32(1) - b2
    decay = f32(1) - f32(lr) * f32(weight_decay)

    def update(pos, m, v):
        gj = g[pos] * coef
        m = m * b1 + omb1 * gj
        v = v * b2 + (omb2 * gj) * gj
        q = p[pos] + step_size * (m / (np.sqrt(v) + eps_bc2))
        if weight_decay > 0:
            q = q * decay
        p[pos] = q
        return m, v

    if blocks8.shape[0]:
        blk, pos, _ = table_positions(blocks8)
        m = st["qmap1"][st["code1"][pos]] * st["absmax1"][blk]
        v = st["qmap2"][st["code2"][pos]] * st["absmax2"][blk]
        m, v = update(pos, m, v)
        starts = np.cumsum(blocks8[:, 1]) - blocks8[:, 1]
        a1, a2 = np.maximum.reduceat(np.abs(m), starts), np.maximum.reduceat(np.abs(v), starts)
        st["absmax1"], st["absmax2"] = a1.astype(f32), a2.astype(f32)
        with np.errstate(divide="ignore", invalid="ignore"):
            x1 = np.where(a1[blk] > 0, m / a1[blk], f32(0)).astype(f32)
            x2 = np.where(a2[blk] > 0, v / a2[blk], f32(0)).astype(f32)
        st["code1"][pos] = quantize(x1, st["qmap1"], m)
        st["code2"][pos] = quantize(x2, st["qmap2"])
    if chunks32.shape[0]:
        _, pos, cpos = table_positions(chunks32)
        st["exp_avg32"][cpos], st["exp_avg_sq32"][cpos] = update(pos, st["exp_avg32"][cpos], st["exp_avg_sq32"][cpos])
    return p, st

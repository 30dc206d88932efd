"""NumPy restatement of torch's dynamic loss-scale update (``torch._amp_update_scale_``, the body of
``GradScaler.update()`` that accelerate runs after every fp16 step, train_online_pso_sdxl_turbo.py:860).  The device
scaler (``pairwise_sample_optimization_b200.amp`` + the ``*_scaled`` boundaries) is checked against it and against torch.

torch's kernel (aten/src/ATen/native/cuda/AmpKernels.cu, ``amp_update_scale_cuda_kernel``; the CPU kernel is the same):

    if found_inf:  scale = scale * backoff_factor ; growth_tracker = 0
    else:          successful = growth_tracker + 1
                   if successful == growth_interval:
                       new_scale = (float)(scale * growth_factor) ; if isfinite(new_scale): scale = new_scale
                       growth_tracker = 0
                   else: growth_tracker = successful

``scale`` is float32, the factors are double: each product is formed in double and rounded to float32.
"""
from __future__ import annotations

import numpy as np


def update_scale(scale: np.float32, growth_tracker: int, found_inf: bool, growth_factor: float, backoff_factor: float,
                 growth_interval: int) -> tuple[np.float32, int]:
    """One ``GradScaler.update()``: returns the new (scale, growth_tracker)."""
    scale = np.float32(scale)
    if found_inf:
        return np.float32(np.float64(scale) * np.float64(backoff_factor)), 0
    successful = int(growth_tracker) + 1
    if successful == growth_interval:
        with np.errstate(over="ignore"):
            grown = np.float32(np.float64(scale) * np.float64(growth_factor))
        return (grown if np.isfinite(grown) else scale), 0
    return scale, successful


def unscale_factor(scale: np.float32) -> np.float32:
    """``GradScaler.unscale_``'s multiplier: ``scale.double().reciprocal().float()``."""
    return np.float32(1.0 / np.float64(np.float32(scale)))

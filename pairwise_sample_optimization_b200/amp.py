"""Dynamic loss scaling for fp16 training with the state on the device (torch's ``GradScaler`` semantics).

The fp16 recipes (train_online_pso_sdxl_turbo.py with ``mixed_precision="fp16"``, :126; the DreamBooth-PSO scripts) run
every step under accelerate's ``GradScaler``: ``scaler.scale(loss).backward()`` (:857), ``unscale_`` + ``clip_grad_norm_``
(:859), ``scaler.step`` + ``scaler.update()`` (:860).  ``DeviceGradScaler`` keeps the scale ``S`` and the growth tracker in
device memory, where the fused kernels read and write them:

* ``pso_pair_loss(..., grad_scaler=s)`` / ``pso_db_loss(..., grad_scaler=s)`` multiply the gradient by ``S`` inside the
  loss kernel, before it is rounded to the prediction dtype (``loss`` and ``stats`` stay unscaled);
* ``FusedLoRAOptimizer(..., grad_scaler=s)`` unscales by ``1 / S`` in its boundary, skips the update when the gradient
  norm is not finite, and updates ``S`` and the tracker at the end of the same launch (``torch._amp_update_scale_``).

So there is no ``update()`` here and no host read anywhere in a step: a step with a scaler can be captured in a CUDA graph.
"""
from __future__ import annotations

import torch

from . import _lib


class DeviceGradScaler:
    """``torch.amp.GradScaler`` state on ``device``, same hyper-parameters and defaults.

    ``scale(loss)`` is ``loss * S`` on the device; ``get_scale()`` reads ``S`` on the host (for logging);
    ``state_dict()`` / ``load_state_dict()`` use torch's format, so the ``scaler.pt`` accelerate saves loads here."""

    def __init__(self, device="cuda", init_scale: float = 2.0 ** 16, growth_factor: float = 2.0,
                 backoff_factor: float = 0.5, growth_interval: int = 2000):
        self.set_hyper(growth_factor, backoff_factor, growth_interval)
        self._scale = torch.full((1,), float(init_scale), dtype=torch.float32, device=device)
        self._growth_tracker = torch.zeros(1, dtype=torch.int32, device=device)
        self.device = self._scale.device  # with the index resolved

    def hyper(self) -> dict:
        return {"growth_factor": self._growth_factor, "backoff_factor": self._backoff_factor,
                "growth_interval": self._growth_interval}

    def set_hyper(self, growth_factor, backoff_factor, growth_interval) -> None:
        if not float(growth_factor) > 1.0:
            raise ValueError(f"growth_factor must be > 1, got {growth_factor}")
        if not 0.0 < float(backoff_factor) < 1.0:
            raise ValueError(f"backoff_factor must be in (0, 1), got {backoff_factor}")
        if int(growth_interval) <= 0:
            raise ValueError(f"growth_interval must be > 0, got {growth_interval}")
        self._growth_factor, self._backoff_factor = float(growth_factor), float(backoff_factor)
        self._growth_interval = int(growth_interval)

    # ---- the step
    def scale(self, loss: torch.Tensor) -> torch.Tensor:
        """``loss * S`` (device multiply, no sync).  ``scale(loss).backward()`` makes the fused losses' upstream factor
        exactly 1: their kernel already scaled the gradient."""
        return loss * self._scale[0]

    def get_scale(self) -> float:
        """The current scale (one host sync: for logging)."""
        return float(self._scale.item())

    @property
    def scale_tensor(self) -> torch.Tensor:
        """``S`` itself (float32[1] on the device), read and written by the kernels."""
        return self._scale

    @property
    def growth_tracker(self) -> torch.Tensor:
        return self._growth_tracker

    def c_struct(self) -> _lib.LossScaler:
        """The ``psob200_loss_scaler`` the ``*_scaled`` entry points take (device pointers + hyper-parameters)."""
        s = _lib.LossScaler()
        s.scale, s.growth_tracker = self._scale.data_ptr(), self._growth_tracker.data_ptr()
        s.growth_factor, s.backoff_factor = self._growth_factor, self._backoff_factor
        s.growth_interval = self._growth_interval
        return s

    # ---- checkpoint (torch.amp.GradScaler.state_dict format)
    def state_dict(self) -> dict:
        return {"scale": self.get_scale(), **self.hyper(), "_growth_tracker": int(self._growth_tracker.item())}

    def load_state_dict(self, state_dict: dict) -> None:
        if len(state_dict) == 0:
            raise RuntimeError("The source state dict is empty, possibly because it was saved from a disabled instance "
                               "of GradScaler.")
        self.set_hyper(state_dict["growth_factor"], state_dict["backoff_factor"], state_dict["growth_interval"])
        self._scale.fill_(float(state_dict["scale"]))
        self._growth_tracker.fill_(int(state_dict["_growth_tracker"]))


def scaler_arg(scaler: DeviceGradScaler, device: torch.device) -> _lib.LossScaler:
    """``scaler``'s C struct, after checking that its state lives on the CUDA device ``device``."""
    if not isinstance(scaler, DeviceGradScaler):
        raise _lib.Psob200Error(f"grad_scaler must be a DeviceGradScaler, got {type(scaler).__name__}")
    idx = device.index if device.index is not None else torch.cuda.current_device()
    if scaler.device.type != "cuda" or scaler.device.index != idx:
        raise _lib.Psob200Error(f"the loss scaler lives on {scaler.device}, the tensors on cuda:{idx}")
    return scaler.c_struct()

"""LoRA adapter checkpoints in the wire format the reference writes (SURVEY.md section 8f rank 2).

The reference's save hook (train_online_pso_sdxl_turbo.py:361-379; dreambooth :1347-1377) runs
``convert_state_dict_to_diffusers(get_peft_model_state_dict(unet))`` and hands the result to
``StableDiffusionXLLoraLoaderMixin.save_lora_weights`` -> ``pytorch_lora_weights.safetensors`` (reloaded at turbo :138).
Those are third-party functions (peft==0.11.1, diffusers==0.27.0; absent here), restated from their published behaviour:

* peft ``get_peft_model_state_dict``: keys ``<module path>.lora_A.weight`` / ``.lora_B.weight`` (adapter name stripped);
* diffusers ``convert_state_dict_to_diffusers`` (PEFT_TO_DIFFUSERS): ``to_q.lora_A`` -> ``to_q.lora.down``,
  ``to_q.lora_B`` -> ``to_q.lora.up`` (same for to_k, to_v, to_out.0);
* ``save_lora_weights``: every key prefixed with ``unet.``, safetensors with metadata ``{"format": "pt"}``.

Parity status: restated, unpinned against the packages.  ``load_lora_weights`` accepts the diffusers keys (with or without
the ``unet.`` prefix) and the peft keys, so files written by either side load.
"""
from __future__ import annotations

import os

import torch

from .lora import LoRALinear

WEIGHT_NAME = "pytorch_lora_weights.safetensors"
OPTIMIZER_NAME = "optimizer.safetensors"  # accelerate writes optimizer.bin next to the model files (save_state, turbo :889)
_TARGETS = ("to_q", "to_k", "to_v", "to_out.0")


def peft_state_dict(model: torch.nn.Module) -> dict:
    """``get_peft_model_state_dict``: adapter tensors keyed by module path, adapter name stripped."""
    out = {}
    for name, m in model.named_modules():
        if isinstance(m, LoRALinear):
            n = m.active_adapter
            out[f"{name}.lora_A.weight"] = m.lora_A[n].weight.detach()
            out[f"{name}.lora_B.weight"] = m.lora_B[n].weight.detach()
    return out


def convert_state_dict_to_diffusers(sd: dict) -> dict:
    out = {}
    for k, v in sd.items():
        for t in _TARGETS:
            k = k.replace(f"{t}.lora_A", f"{t}.lora.down").replace(f"{t}.lora_B", f"{t}.lora.up")
        out[k] = v
    return out


def convert_state_dict_to_peft(sd: dict) -> dict:
    out = {}
    for k, v in sd.items():
        if k.startswith("unet."):
            k = k[len("unet."):]
        out[k.replace(".lora.down.", ".lora_A.").replace(".lora.up.", ".lora_B.")] = v
    return out


def save_lora_weights(save_directory: str, unet: torch.nn.Module, weight_name: str = WEIGHT_NAME) -> str:
    """Write the adapters of ``unet`` as ``<save_directory>/pytorch_lora_weights.safetensors`` (diffusers key naming)."""
    from safetensors.torch import save_file
    os.makedirs(save_directory, exist_ok=True)
    sd = {f"unet.{k}": v.to("cpu").contiguous() for k, v in convert_state_dict_to_diffusers(peft_state_dict(unet)).items()}
    path = os.path.join(save_directory, weight_name)
    save_file(sd, path, metadata={"format": "pt"})
    return path


def load_lora_weights(path: str, unet: torch.nn.Module, strict: bool = True) -> list:
    """Load adapters written by ``save_lora_weights`` (or by the reference's hook) into the ``LoRALinear`` modules of
    ``unet``.  Returns the list of loaded keys; ``strict`` raises on missing / unexpected / mis-shaped tensors."""
    from safetensors.torch import load_file
    if os.path.isdir(path):
        path = os.path.join(path, WEIGHT_NAME)
    sd = convert_state_dict_to_peft(load_file(path))
    mods = {name: m for name, m in unet.named_modules() if isinstance(m, LoRALinear)}
    loaded, missing = [], []
    for name, m in mods.items():
        n = m.active_adapter
        for which, lin in (("lora_A", m.lora_A[n]), ("lora_B", m.lora_B[n])):
            key = f"{name}.{which}.weight"
            if key not in sd:
                missing.append(key)
                continue
            t = sd.pop(key)
            if tuple(t.shape) != tuple(lin.weight.shape):
                raise ValueError(f"{key}: checkpoint shape {tuple(t.shape)} != adapter shape {tuple(lin.weight.shape)} "
                                 "(different LoRA rank?)")
            with torch.no_grad():
                lin.weight.copy_(t.to(device=lin.weight.device, dtype=lin.weight.dtype))
            loaded.append(key)
    if strict and (missing or sd):
        raise KeyError(f"missing keys: {missing[:4]}{'...' if len(missing) > 4 else ''}; "
                       f"unexpected keys: {list(sd)[:4]}{'...' if len(sd) > 4 else ''}")
    return loaded


# ----------------------------------------------------------------------------------------------- optimizer state
def save_optimizer_state(save_directory: str, optimizer, name: str = OPTIMIZER_NAME) -> str:
    """The resumable part of ``accelerator.save_state`` (turbo :886-889) for ``lora.FusedLoRAOptimizer``: fp32 master
    parameters, both AdamW moments, the count of applied updates and the hyper-parameters, in one safetensors file.
    Every tensor of ``optimizer.state_dict()`` is stored as a tensor and every other entry as JSON metadata, so the 8-bit
    state (uint8 codes, absmax arrays, compact fp32 moments, both maps, and the keys that describe its format) travels
    the same way."""
    import json
    from safetensors.torch import save_file
    os.makedirs(save_directory, exist_ok=True)
    sd = optimizer.state_dict()
    tensors = {k: v.to("cpu").contiguous() for k, v in sd.items() if isinstance(v, torch.Tensor)}
    meta = {"format": "pt", **{k: json.dumps(v) for k, v in sd.items() if not isinstance(v, torch.Tensor)}}
    path = os.path.join(save_directory, name)
    save_file(tensors, path, metadata=meta)
    return path


def load_optimizer_state(path: str, optimizer, load_hyper: bool = True) -> None:
    """Inverse of ``save_optimizer_state`` (``accelerator.load_state`` through the hook registered at turbo :398): restores moments, step count and the
    master parameters (hence the adapters and their 16-bit operand copies)."""
    import json
    from safetensors import safe_open
    if os.path.isdir(path):
        path = os.path.join(path, OPTIMIZER_NAME)
    with safe_open(path, framework="pt", device="cpu") as f:
        meta = f.metadata()
        sd = {k: f.get_tensor(k) for k in f.keys()}
    sd.update({k: json.loads(v) for k, v in meta.items() if k != "format"})
    optimizer.load_state_dict(sd, load_hyper=load_hyper)


def save_state(save_directory: str, unet: torch.nn.Module, optimizer=None) -> None:
    """``accelerator.save_state(dir)`` as the trainers use it (turbo :886-889): adapters in the diffusers wire format (the
    save hook, :361-379) and, next to them, the optimizer state."""
    save_lora_weights(save_directory, unet)
    if optimizer is not None:
        save_optimizer_state(save_directory, optimizer)


def load_state(save_directory: str, unet: torch.nn.Module, optimizer=None) -> None:
    """``accelerator.load_state(dir)``.  With an optimizer its fp32 master parameters win (they ARE the adapters); without,
    only the adapter file is read."""
    load_lora_weights(save_directory, unet)
    if optimizer is not None:
        load_optimizer_state(save_directory, optimizer)

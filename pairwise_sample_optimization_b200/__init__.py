"""pairwise_sample_optimization_b200 -- the B200-native (sm_100a) PSO training-step hot path.

Only what the path needs (SURVEY.md section 8):

* ``csrc/`` + ``libpsob200.so``  hand-written CUDA kernels behind the C ABI of ``include/psob200.h``
* ``pso_pytorch.diffusers_patch`` drop-ins for the reference's step / sampler functions (same names)
* ``losses``                      fused online-PSO and DreamBooth-PSO loss + gradient
* ``lora`` / ``gemm``              LoRA-wrapped attention projections (peft / diffusers surface) on the tcgen05 GEMM kernels
* ``feed_forward``                fused gated GELU (GEGLU) of the transformer feed-forward, forward + backward
* ``checkpoint``                  LoRA adapters in the reference's safetensors wire format (+ optimizer state)
* ``reward_preprocess``           decoded images -> CLIP / PickScore ``pixel_values`` on the device (Pillow-exact resize)
* ``runtime``                     device-resident schedule tables, workspace, status word
* ``amp``                         fp16 dynamic loss scaling with the scale on the device (GradScaler semantics)

There is no CPU or PyTorch fallback: every op raises if the CUDA library is missing.
"""
from . import _lib, amp, checkpoint, feed_forward, gemm, lora, reward_preprocess, runtime
from .amp import DeviceGradScaler
from .losses import compare, edm_sigmas, pso_db_loss, pso_pair_loss, sample_compare
from .pso_pytorch.diffusers_patch import (
    _get_x0_from_noise,
    distilled_step_with_logprob,
    sdxl_dmd_pipeline_with_logprob,
    sdxl_turbo_pipeline_with_logprob,
    turbo_step_with_logprob,
)
from .reward_preprocess import DeviceCLIPImageProcessor, clip_image_preprocess
from .runtime import check_status

__all__ = [
    "turbo_step_with_logprob",
    "distilled_step_with_logprob",
    "_get_x0_from_noise",
    "sdxl_turbo_pipeline_with_logprob",
    "sdxl_dmd_pipeline_with_logprob",
    "pso_pair_loss",
    "pso_db_loss",
    "edm_sigmas",
    "sample_compare",
    "compare",
    "check_status",
    "clip_image_preprocess",
    "DeviceCLIPImageProcessor",
    "DeviceGradScaler",
]

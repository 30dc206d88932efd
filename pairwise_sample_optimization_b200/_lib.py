"""ctypes binding of the C ABI declared in include/psob200.h.

The product path has NO fallback: if ``libpsob200.so`` is missing or does not export a
symbol, importing this module's ``lib()`` raises; every op then fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os

import torch

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG_DIR, "libpsob200.so")

F32, BF16, F16, U8 = 0, 1, 2, 3
TS_I64, TS_F32, TS_I32 = 0, 1, 2
SCHED_TURBO, SCHED_DMD, SCHED_AFFINE = 0, 1, 2
DB_PSO, DB_PSO_DB = 0, 1
STATUS_TIMESTEP_NOT_IN_SCHEDULE = 1
STATUS_NONFINITE_COEFFICIENT = 2

_DTYPES = {torch.float32: F32, torch.bfloat16: BF16, torch.float16: F16}
_TS_DTYPES = {torch.int64: TS_I64, torch.float32: TS_F32, torch.int32: TS_I32}

_vp, _fp, _ip = C.c_void_p, C.c_void_p, C.c_void_p  # all device pointers travel as integers


class Schedule(C.Structure):
    _fields_ = [("kind", C.c_int32), ("n_table", C.c_int32), ("sched_timesteps", _fp), ("table", _fp),
                ("ts_dtype", C.c_int32), ("reserved", C.c_int32)]


class OnlinePsoArgs(C.Structure):
    _fields_ = [("pred", _vp * 2), ("ref", _vp * 2), ("sample", _vp * 2), ("next", _vp * 2), ("ts", _vp * 2),
                ("ts_prev", _vp * 2), ("coef", _fp * 2), ("human_prefer", _fp),
                ("stride_pred", C.c_int64 * 2), ("stride_ref", C.c_int64 * 2), ("stride_sample", C.c_int64 * 2),
                ("stride_next", C.c_int64 * 2), ("grad", _vp * 2), ("loss", _fp), ("stats", _fp), ("status", _ip),
                ("workspace", _vp), ("workspace_bytes", C.c_size_t), ("B", C.c_int64), ("N", C.c_int64),
                ("pred_dtype", C.c_int32), ("latent_dtype", C.c_int32), ("beta", C.c_float), ("eps", C.c_float),
                ("loss_scale", C.c_float), ("tune_threads", C.c_int32), ("tune_cluster", C.c_int32),
                ("reserved", C.c_int32)]


class DreamboothArgs(C.Structure):
    _fields_ = [("model_pred", _vp), ("ref_pred", _vp), ("noisy", _vp), ("target", _vp), ("sigmas", _fp),
                ("grad", _vp), ("loss", _fp), ("stats", _fp), ("status", _ip), ("workspace", _vp),
                ("workspace_bytes", C.c_size_t), ("b", C.c_int64), ("N", C.c_int64), ("pred_dtype", C.c_int32),
                ("latent_dtype", C.c_int32), ("loss_type", C.c_int32), ("beta_pso", C.c_float),
                ("neg_defactor", C.c_float), ("prior_loss_weight", C.c_float), ("loss_scale", C.c_float),
                ("tune_threads", C.c_int32), ("tune_cluster", C.c_int32), ("reserved", C.c_int32)]


class StepArgs(C.Structure):
    _fields_ = [("model_output", _vp), ("sample", _vp), ("prev_sample", _vp), ("noise", _vp), ("ts", _vp),
                ("ts_prev", _vp), ("coef", _fp), ("prev_out", _vp), ("scaled_next_out", _vp), ("log_prob", _fp),
                ("status", _ip), ("B", C.c_int64), ("N", C.c_int64), ("noise_rows", C.c_int64),
                ("ts_rows", C.c_int64), ("stride_model_output", C.c_int64), ("stride_sample", C.c_int64),
                ("stride_prev_sample", C.c_int64), ("pred_dtype", C.c_int32), ("latent_dtype", C.c_int32),
                ("out_dtype", C.c_int32), ("tune_threads", C.c_int32), ("tune_cluster", C.c_int32),
                ("use_philox", C.c_int32), ("philox_seed", C.c_uint64), ("philox_offset", C.c_uint64)]


class StepBwdArgs(C.Structure):
    _fields_ = [("model_output", _vp), ("sample", _vp), ("prev_sample", _vp), ("ts", _vp), ("ts_prev", _vp),
                ("coef", _fp), ("grad_log_prob", _fp), ("grad_model_output", _vp), ("status", _ip),
                ("B", C.c_int64), ("N", C.c_int64), ("ts_rows", C.c_int64), ("stride_model_output", C.c_int64),
                ("stride_sample", C.c_int64), ("stride_prev_sample", C.c_int64), ("pred_dtype", C.c_int32),
                ("latent_dtype", C.c_int32), ("reserved0", C.c_int32), ("reserved1", C.c_int32)]


class GemmArgs(C.Structure):
    _fields_ = [("a1", _vp), ("b1", _vp), ("a2", _vp), ("b2", _vp), ("bias", _vp), ("d", _vp), ("dt", _vp),
                ("lda1", C.c_int64), ("ldb1", C.c_int64), ("lda2", C.c_int64), ("ldb2", C.c_int64),
                ("ldd", C.c_int64), ("lddt", C.c_int64), ("M", C.c_int64), ("N", C.c_int64), ("K1", C.c_int64),
                ("K2", C.c_int64), ("alpha", C.c_float), ("ab_dtype", C.c_int32), ("d_dtype", C.c_int32),
                ("bias_dtype", C.c_int32), ("a_reduction_major", C.c_int32), ("b_reduction_major", C.c_int32),
                ("accumulate", C.c_int32),
                ("split_k", C.c_int32), ("tune_bn", C.c_int32), ("pdl", C.c_int32), ("diag", C.c_int32)]


class LoraLinearArgs(C.Structure):
    _fields_ = [("x", _vp), ("w", _vp), ("bias", _vp), ("lora_a", _vp), ("lora_b", _vp), ("y", _vp), ("t", _vp),
                ("tt", _vp), ("dy", _vp), ("dx", _vp), ("u", _vp), ("ut", _vp), ("d_lora_a", _fp), ("d_lora_b", _fp),
                ("ldx", C.c_int64), ("ldw", C.c_int64), ("lda", C.c_int64), ("ldb", C.c_int64), ("ldy", C.c_int64),
                ("ldt", C.c_int64), ("ldtt", C.c_int64), ("lddy", C.c_int64), ("lddx", C.c_int64),
                ("ldu", C.c_int64), ("ldut", C.c_int64), ("ld_da", C.c_int64), ("ld_db", C.c_int64),
                ("M", C.c_int64), ("K", C.c_int64), ("N", C.c_int64), ("r", C.c_int64), ("scaling", C.c_float),
                ("dtype", C.c_int32), ("bias_dtype", C.c_int32), ("adapters_enabled", C.c_int32),
                ("backward_phases", C.c_int32), ("forward_phases", C.c_int32), ("flags", _vp), ("flags_len", C.c_int64)]


class LoraGroupArgs(C.Structure):
    _fields_ = [("x", _vp), ("w", _vp), ("bias", _vp), ("lora_a", _vp), ("lora_b", _vp), ("y", _vp), ("t", _vp), ("tt", _vp),
                ("dy", _vp * 3), ("dx", _vp), ("u", _vp), ("ut", _vp), ("d_lora_a", _fp), ("d_lora_b", _fp), ("flags", _vp),
                ("flags_len", C.c_int64), ("ldx", C.c_int64), ("ldw", C.c_int64), ("lda", C.c_int64), ("ldb", C.c_int64),
                ("ldy", C.c_int64), ("ldt", C.c_int64), ("ldtt", C.c_int64), ("lddy", C.c_int64 * 3), ("lddx", C.c_int64),
                ("ldu", C.c_int64), ("ldut", C.c_int64), ("ld_da", C.c_int64), ("ld_db", C.c_int64), ("M", C.c_int64),
                ("K", C.c_int64), ("N", C.c_int64), ("r", C.c_int64), ("G", C.c_int32), ("scaling", C.c_float),
                ("dtype", C.c_int32), ("bias_dtype", C.c_int32), ("adapters_enabled", C.c_int32),
                ("forward_phases", C.c_int32), ("backward_phases", C.c_int32), ("launch_flags", C.c_int32),
                ("r_stride", C.c_int64)]


class FlatAdamwArgs(C.Structure):
    _fields_ = [("param", _fp), ("grad", _fp), ("exp_avg", _fp), ("exp_avg_sq", _fp), ("operand", _vp), ("norm_out", _fp),
                ("workspace", _vp), ("n", C.c_int64), ("step", C.c_int64), ("lr", C.c_float), ("beta1", C.c_float),
                ("beta2", C.c_float), ("eps", C.c_float), ("weight_decay", C.c_float), ("max_grad_norm", C.c_float),
                ("grad_scale", C.c_float), ("operand_dtype", C.c_int32), ("n_sumsq_parts", C.c_int32), ("sumsq_parts", _vp),
                ("found_inf", _fp), ("step_dev", _vp)]


class FlatAdamw8Args(C.Structure):
    _fields_ = [("param", _fp), ("grad", _fp), ("code1", _vp), ("code2", _vp), ("absmax1", _fp), ("absmax2", _fp),
                ("map1", _fp), ("map2", _fp), ("blocks8", _vp), ("n_blocks8", C.c_int64), ("chunks32", _vp),
                ("n_chunks32", C.c_int64), ("exp_avg32", _fp), ("exp_avg_sq32", _fp), ("operand", _vp), ("norm_out", _fp),
                ("workspace", _vp), ("n", C.c_int64), ("step", C.c_int64), ("lr", C.c_float), ("beta1", C.c_float),
                ("beta2", C.c_float), ("eps", C.c_float), ("weight_decay", C.c_float), ("max_grad_norm", C.c_float),
                ("grad_scale", C.c_float), ("operand_dtype", C.c_int32), ("n_sumsq_parts", C.c_int32),
                ("block_size", C.c_int32), ("sumsq_parts", _vp), ("found_inf", _fp), ("step_dev", _vp)]


class LossScaler(C.Structure):
    _fields_ = [("scale", _fp), ("growth_tracker", _ip), ("growth_factor", C.c_double), ("backoff_factor", C.c_double),
                ("growth_interval", C.c_int32), ("reserved", C.c_int32)]


class FlatAllreduceArgs(C.Structure):
    _fields_ = [("grad_multicast", _vp), ("sumsq_multicast", _vp), ("n", C.c_int64), ("rank", C.c_int32),
                ("world", C.c_int32), ("scale", C.c_float)]


class GegluArgs(C.Structure):
    _fields_ = [("proj", _vp), ("out", _vp), ("dout", _vp), ("dproj", _vp), ("M", C.c_int64), ("I", C.c_int64),
                ("ld_proj", C.c_int64), ("ld_out", C.c_int64), ("ld_dout", C.c_int64), ("ld_dproj", C.c_int64),
                ("dtype", C.c_int32)]


class ClipPreprocessArgs(C.Structure):
    _fields_ = [("src", _vp), ("dst", _vp), ("bounds_h", _vp), ("coeffs_h", _vp), ("bounds_v", _vp), ("coeffs_v", _vp),
                ("norm_table", _fp), ("B", C.c_int64), ("in_h", C.c_int64), ("in_w", C.c_int64), ("rs_h", C.c_int64),
                ("rs_w", C.c_int64), ("out_h", C.c_int64), ("out_w", C.c_int64), ("crop_top", C.c_int64),
                ("crop_left", C.c_int64), ("taps_h", C.c_int32), ("taps_v", C.c_int32), ("src_dtype", C.c_int32),
                ("dst_dtype", C.c_int32)]


class LayerNormArgs(C.Structure):
    _fields_ = [("x", _vp), ("y", _vp), ("dy", _vp), ("dx", _vp), ("weight", _vp), ("bias", _vp), ("mean", _fp), ("rstd", _fp),
                ("rows", C.c_int64), ("C", C.c_int64), ("ld_x", C.c_int64), ("ld_y", C.c_int64), ("ld_dy", C.c_int64),
                ("ld_dx", C.c_int64), ("eps", C.c_float), ("dtype", C.c_int32), ("out_dtype", C.c_int32),
                ("param_dtype", C.c_int32)]


class GroupNormArgs(C.Structure):
    _fields_ = [("x", _vp), ("channel_add", _vp), ("y", _vp), ("dy", _vp), ("dx", _vp), ("weight", _vp), ("bias", _vp),
                ("mean", _fp), ("rstd", _fp), ("workspace", _vp), ("workspace_bytes", C.c_size_t), ("N", C.c_int64),
                ("C", C.c_int64), ("HW", C.c_int64), ("G", C.c_int32), ("eps", C.c_float), ("dtype", C.c_int32),
                ("out_dtype", C.c_int32), ("param_dtype", C.c_int32), ("silu", C.c_int32)]


_STRUCTS = {0: Schedule, 1: OnlinePsoArgs, 2: DreamboothArgs, 3: StepArgs, 4: StepBwdArgs, 5: GemmArgs,
            6: LoraLinearArgs, 7: FlatAdamwArgs, 8: GegluArgs, 9: FlatAllreduceArgs, 10: ClipPreprocessArgs, 11: LoraGroupArgs,
            12: FlatAdamw8Args, 13: LossScaler, 14: LayerNormArgs, 15: GroupNormArgs}

# name -> (restype, argtypes): every symbol include/psob200.h declares
SIGNATURES = {
    "psob200_abi_version": (C.c_int, []),
    "psob200_strerror": (C.c_char_p, [C.c_int]),
    "psob200_last_error_detail": (C.c_char_p, []),
    "psob200_device_sm_count": (C.c_int, []),
    "psob200_launch_count": (C.c_longlong, []),
    "psob200_struct_size": (C.c_size_t, [C.c_int]),
    "psob200_pair_loss_workspace_bytes": (C.c_size_t, [C.c_int64]),
    "psob200_online_pso_loss_grad": (C.c_int, [C.POINTER(Schedule), C.POINTER(OnlinePsoArgs), _vp]),
    "psob200_dreambooth_pso_loss_grad": (C.c_int, [C.POINTER(DreamboothArgs), _vp]),
    "psob200_online_pso_loss_grad_scaled": (C.c_int, [C.POINTER(Schedule), C.POINTER(OnlinePsoArgs), C.POINTER(LossScaler),
                                                      _vp]),
    "psob200_dreambooth_pso_loss_grad_scaled": (C.c_int, [C.POINTER(DreamboothArgs), C.POINTER(LossScaler), _vp]),
    "psob200_step_logprob": (C.c_int, [C.POINTER(Schedule), C.POINTER(StepArgs), _vp]),
    "psob200_step_logprob_backward": (C.c_int, [C.POINTER(Schedule), C.POINTER(StepBwdArgs), _vp]),
    "psob200_dmd_x0_from_noise": (C.c_int, [_fp, C.c_int32, _vp, _vp, _vp, C.c_int32, C.c_int64, _vp, C.c_int64,
                                            C.c_int64, C.c_int32, C.c_int32, C.c_int32, _ip, _vp]),
    "psob200_lora_gemm": (C.c_int, [C.POINTER(GemmArgs), _vp]),
    "psob200_lora_gemm_timeline": (C.c_int, [C.POINTER(C.c_ulonglong), C.c_longlong]),
    "psob200_lora_linear_forward": (C.c_int, [C.POINTER(LoraLinearArgs), _vp]),
    "psob200_lora_linear_backward": (C.c_int, [C.POINTER(LoraLinearArgs), _vp]),
    "psob200_lora_group_forward": (C.c_int, [C.POINTER(LoraGroupArgs), _vp]),
    "psob200_lora_group_backward": (C.c_int, [C.POINTER(LoraGroupArgs), _vp]),
    "psob200_flat_adamw_step": (C.c_int, [C.POINTER(FlatAdamwArgs), _vp]),
    "psob200_flat_adamw8_step": (C.c_int, [C.POINTER(FlatAdamw8Args), _vp]),
    "psob200_flat_adamw_step_scaled": (C.c_int, [C.POINTER(FlatAdamwArgs), C.POINTER(LossScaler), _vp]),
    "psob200_flat_adamw8_step_scaled": (C.c_int, [C.POINTER(FlatAdamw8Args), C.POINTER(LossScaler), _vp]),
    "psob200_flat_allreduce_sumsq": (C.c_int, [C.POINTER(FlatAllreduceArgs), _vp]),
    "psob200_geglu_forward": (C.c_int, [C.POINTER(GegluArgs), _vp]),
    "psob200_geglu_backward": (C.c_int, [C.POINTER(GegluArgs), _vp]),
    "psob200_layer_norm_forward": (C.c_int, [C.POINTER(LayerNormArgs), _vp]),
    "psob200_layer_norm_backward": (C.c_int, [C.POINTER(LayerNormArgs), _vp]),
    "psob200_group_norm_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int64, C.c_int64, C.c_int32]),
    "psob200_group_norm_forward": (C.c_int, [C.POINTER(GroupNormArgs), _vp]),
    "psob200_group_norm_backward": (C.c_int, [C.POINTER(GroupNormArgs), _vp]),
    "psob200_resample_taps": (C.c_int, [C.c_int64, C.c_int64]),
    "psob200_resample_plan": (C.c_int, [C.c_int64, C.c_int64, C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "psob200_clip_norm_table": (C.c_int, [C.c_double, C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_float)]),
    "psob200_clip_preprocess": (C.c_int, [C.POINTER(ClipPreprocessArgs), _vp]),
    "psob200_scale": (C.c_int, [_vp, _vp, C.c_int64, C.c_float, C.c_int32, C.c_int32, _vp]),
    "psob200_scale_inplace_by_device_scalar": (C.c_int, [_vp, C.c_int64, C.c_int32, _fp, _vp]),
}

_lib = None


class Psob200Error(RuntimeError):
    pass


def lib() -> C.CDLL:
    """Load libpsob200.so (once) and bind every declared symbol.  Raises if anything is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise Psob200Error(
            f"{LIB_PATH} not found: build it with `python -m pairwise_sample_optimization_b200.build` "
            "(there is no CPU or PyTorch fallback for the PSO hot path)")
    handle = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(handle, name)  # AttributeError if the library does not export it
        fn.restype = res
        fn.argtypes = args
    for which, struct in _STRUCTS.items():
        got = handle.psob200_struct_size(which)
        if got != C.sizeof(struct):
            raise Psob200Error(f"ABI mismatch: {struct.__name__} is {C.sizeof(struct)} bytes here, {got} in the library")
    _lib = handle
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        detail = lib().psob200_last_error_detail().decode() if rc == -4 else ""
        raise Psob200Error(f"{what} failed: {lib().psob200_strerror(rc).decode()} (rc={rc}){' -- ' + detail if detail else ''}")


def dtype_code(t: torch.Tensor) -> int:
    try:
        return _DTYPES[t.dtype]
    except KeyError:
        raise Psob200Error(f"unsupported element type {t.dtype} (float32, bfloat16, float16 only)") from None


def ts_dtype_code(t: torch.Tensor) -> int:
    return _TS_DTYPES[t.dtype]


def require_cuda(*tensors: torch.Tensor) -> torch.device:
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise Psob200Error("the PSO hot path runs on a CUDA device only (no CPU fallback); got a "
                               f"{t.device} tensor")
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise Psob200Error(f"tensors on different devices: {dev} and {t.device}")
    return dev


class _NoGuard:
    def __enter__(self):
        return None

    def __exit__(self, *exc):
        return False


_NO_GUARD = _NoGuard()


def on_device(device: torch.device):
    """Context for a C-ABI call: the library launches on the calling thread's CURRENT device (and keys its per-device
    caches by it), so a call on tensors of another device must switch first.  Free when the device is already current."""
    idx = device.index if device.index is not None else torch.cuda.current_device()
    return _NO_GUARD if idx == torch.cuda.current_device() else torch.cuda.device(idx)


def launch(device: torch.device, name: str, *args) -> None:
    """One C-ABI call on ``device`` (made current for the call if it is not), raising on a non-zero return code."""
    with on_device(device):
        rc = getattr(lib(), name)(*args)
    check(rc, name)


def current_stream(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def rows(t: torch.Tensor, n: int) -> tuple[torch.Tensor, int]:
    """View ``t`` as [B, N] rows without copying when each sample is dense; returns (tensor, row stride)."""
    B = t.shape[0]
    if t.dim() >= 2 and t[0].is_contiguous() and (B == 1 or t.stride(0) >= n):
        return t, (t.stride(0) if B > 1 else n)
    t = t.contiguous()
    return t, n

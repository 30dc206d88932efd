#!/usr/bin/env python
"""The optimizer boundary alone, fp32 AdamW (psob200_flat_adamw_step) against blockwise 8-bit AdamW
(psob200_flat_adamw8_step), over the flat LoRA layout of the SDXL UNet (1 120 adapter matrices) at r = 8 and r = 64.

    python tools/bench_flat_optimizer.py [--iters 50] [--warmup 10] [--scaler]

Prints one JSON line.  Each timed boundary is bracketed by CUDA events; the gradient is rewritten with fresh values before
every boundary (outside the events), as the backward would leave it.  "norm included" = norm launch + update launch (what
step() does after an NCCL exchange); "norm supplied" = the update launch alone (after the fused multimem exchange, which
delivers the sum of squares).  GB/s are algorithmic bytes over event time:
  fp32: norm 4 B/param; update reads p, g, m, v and writes p, m, v, g (32 B) + the 16-bit operand (2 B)
  8-bit: norm 4 B/param; update reads / writes p and g (16 B), reads / writes two 1-byte codes (4 B) + the operand (2 B)
(absmax arrays: 16 B per 256-element block, not counted).
--scaler: each boundary is also run with a device loss scaler attached (psob200_flat_adamw*_step_scaled), alternating
with the unscaled one in the same loop; "norm_*_scaler" holds its times next to the unscaled "norm_*"."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from fixtures import sdxl_unet  # noqa: E402
from pairwise_sample_optimization_b200 import _lib, amp, lora  # noqa: E402

BYTES = {32: {"included": 38, "supplied": 34}, 8: {"included": 26, "supplied": 22}}


def sdxl_projections():
    with torch.device("meta"):
        unet = sdxl_unet.UNet2DConditionModel(sdxl_unet.sdxl_config())
    return [(m.in_features, m.out_features) for n, m in unet.named_modules()
            if isinstance(m, torch.nn.Linear) and n.endswith((".to_q", ".to_k", ".to_v", ".to_out.0"))]


def build(shapes, r, bits, dev):
    model = torch.nn.ModuleList()
    for k, n in shapes:
        lay = lora.LoRALinear(torch.nn.Linear(k, n, bias=False, device=dev, dtype=torch.bfloat16), r, r)
        torch.nn.init.normal_(lay.lora_B["default"].weight, std=0.02)
        model.append(lay)
    return lora.FusedLoRAOptimizer(model, lr=1e-4, weight_decay=1e-2, max_grad_norm=1.0, optim_bits=bits)


def time_boundary(opt, norm, iters, warmup, dev, scalers=(None,)):
    """(median ms, min ms) of the boundary for each entry of `scalers` (None = no loss scaler), the variants alternating
    boundary by boundary on the same optimizer and gradients."""
    parts = torch.zeros(1, dtype=torch.float64, device=dev)
    grads = [torch.randn(opt.bucket.flat.numel(), device=dev, generator=torch.Generator(device=dev).manual_seed(s)) * 1e-3
             for s in range(2)]
    stream = _lib.current_stream(dev)
    times = [[] for _ in scalers]
    for i in range(warmup + iters):
        for v, sc in enumerate(scalers):
            opt.grad_scaler = sc
            opt.bucket.flat.copy_(grads[i % 2])
            entry, a, extra = opt._launch_args()
            if norm == "supplied":
                parts.fill_(1e-2)
                a.n_sumsq_parts, a.sumsq_parts = 1, parts.data_ptr()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            _lib.launch(dev, entry, C.byref(a), *extra, stream)
            e1.record()
            if i >= warmup:
                times[v].append((e0, e1))
    opt.grad_scaler = None
    torch.cuda.synchronize()
    assert float(opt.found_inf) == 0.0 and float(opt.bucket.flat.abs().max()) == 0.0
    out = []
    for t in times:
        ms = sorted(e0.elapsed_time(e1) for e0, e1 in t)
        out.append((ms[len(ms) // 2], ms[0]))
    return out if len(scalers) > 1 else out[0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--scaler", action="store_true",
                    help="also time every boundary with a DeviceGradScaler attached (the *_scaled entry points), alternating "
                         "with the unscaled boundary in the same loop")
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    _lib.lib()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    peaks = os.path.join(ROOT, "MEASURED_PEAKS.json")
    hbm = json.load(open(peaks))["hbm_gbs"] if os.path.exists(peaks) else None
    shapes = sdxl_projections()
    out = {"tool": "bench_flat_optimizer", "gpu": gpu, "hbm_copy_peak_gbs": hbm,
           "hbm_copy_peak_source": "MEASURED_PEAKS.json" if hbm else None, "iters": args.iters, "ranks": []}
    for r in (8, 64):
        entry = {"r": r}
        for bits in (32, 8):
            opt = build(shapes, r, bits, dev)
            n = sum(p.numel() for p in opt.bucket.params)
            entry["params"], entry["matrices"] = n, len(opt.bucket.params)
            if bits == 32:
                state = opt.exp_avg.numel() * 4 * 2
            else:
                state = sum(t.numel() * t.element_size() for t in (opt.code1, opt.code2, opt.absmax1, opt.absmax2,
                                                                   opt.exp_avg32, opt.exp_avg_sq32))
                entry["blocks8"], entry["fp32_class_elements"] = int(opt.blocks8.shape[0]), int(opt.exp_avg32.numel())
            res = {"state_mb": round(state / 1e6, 1)}
            for norm in ("included", "supplied"):
                if args.scaler:  # S = 1 and an interval that is never reached: the same arithmetic, the scaled launch
                    sc = amp.DeviceGradScaler(dev, init_scale=1.0, growth_interval=2 ** 30)
                    (med, best), (med_s, best_s) = time_boundary(opt, norm, args.iters, args.warmup, dev, (None, sc))
                    res[f"norm_{norm}_scaler"] = {"median_ms": round(med_s, 4), "min_ms": round(best_s, 4),
                                                  "ratio_over_unscaled": round(med_s / med, 3)}
                else:
                    med, best = time_boundary(opt, norm, args.iters, args.warmup, dev)
                res[f"norm_{norm}"] = {"median_ms": round(med, 4), "min_ms": round(best, 4), "bytes_per_param": BYTES[bits][norm],
                                       "gbs": round(BYTES[bits][norm] * n / (med * 1e-3) / 1e9, 1)}
            entry[f"adamw{bits}"] = res
            del opt
            torch.cuda.empty_cache()
        for norm in ("included", "supplied"):
            entry[f"ratio_8_over_32_norm_{norm}"] = round(entry["adamw8"][f"norm_{norm}"]["median_ms"] /
                                                          entry["adamw32"][f"norm_{norm}"]["median_ms"], 3)
        out["ranks"].append(entry)
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()

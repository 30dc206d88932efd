#!/usr/bin/env python
"""Fused norms (norms.install_fused_norms) against stock torch, on one B200:

1. every norm shape of the dmd128 and turbo64 micro-steps at batch 8 (2 x 4 pairs, bf16): F.layer_norm / F.group_norm
   (+ F.silu, + the broadcast time-embedding add of ResnetBlock2D) vs the fused kernels, forward alone and backward
   (= forward + backward minus forward), CUDA events around CUDA-graph replays.  Each replay walks through enough input
   copies to stream >= 256 MB, so the inputs come from HBM, not from the 126 MB L2.  Bytes are algorithmic (each tensor the
   op must read or write, once), GB/s = bytes / time.
2. the graph-replayed micro-step of bench.py (its B200Arm: batched forwards, second-stream reference, fused GEGLU,
   deterministic mode) without and with install_fused_norms, the two arms alternated in one process; ms/step and the peak
   memory of one eager micro-step of each arm.
3. the card name and power limit, read in the same run.

    python tools/bench_norms.py [--configs dmd128,turbo64] [--reps 20] [--steps 10] [--rounds 3] [--json OUT]
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys

import torch
import torch.nn as nn
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from fixtures import micro_step, sdxl_unet  # noqa: E402

STREAM_BYTES = 256 << 20


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        out = f"nvidia-smi unavailable ({e})"
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": out}


def norm_shapes(hw, batch):
    """(kind, shape, groups, eps) -> count for one forward of the SDXL fixture, found by running it on the meta device."""
    cfg = sdxl_unet.sdxl_config()
    with torch.device("meta"):
        unet = sdxl_unet.UNet2DConditionModel(cfg)
    found = {}
    parents = {}
    for name, m in unet.named_modules():
        for cname, c in m.named_children():
            parents[c] = (m, cname)

    def hook(mod, args, _out):
        x = args[0]
        if isinstance(mod, nn.LayerNorm):
            key = ("layer_norm", (math.prod(x.shape[:-1]), x.shape[-1]), 0, mod.eps)
        else:
            parent, cname = parents[mod]
            kind = "group_norm"
            if type(parent).__name__ == "ResnetBlock2D":
                kind = "group_norm+silu" if cname == "norm1" else "group_norm+add+silu"
            key = (kind, tuple(x.shape), mod.num_groups, mod.eps)
        found[key] = found.get(key, 0) + 1

    for m in unet.modules():
        if isinstance(m, (nn.LayerNorm, nn.GroupNorm)):
            m.register_forward_hook(hook)
    pooled = cfg.projection_class_embeddings_input_dim - 6 * cfg.addition_time_embed_dim
    with torch.device("meta"):
        unet(torch.empty(batch, 4, hw, hw), torch.full((batch,), 999), torch.empty(batch, 77, cfg.cross_attention_dim),
             added_cond_kwargs={"text_embeds": torch.empty(batch, pooled), "time_ids": torch.empty(batch, 6)})
    return found


def timed(fn, reps):
    """Median device time (us) of one graph replay of ``fn``."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=side):
        fn()
    for _ in range(2):
        graph.replay()
    torch.cuda.synchronize()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in evs:
        a.record()
        graph.replay()
        b.record()
    torch.cuda.synchronize()
    return statistics.median(a.elapsed_time(b) for a, b in evs) * 1e3


def per_shape(norms, key, reps):
    kind, shape, groups, eps = key
    dt, dev = torch.bfloat16, torch.device("cuda", 0)
    xbytes = math.prod(shape) * 2
    copies = max(2, math.ceil(STREAM_BYTES / xbytes))
    c = shape[-1] if kind == "layer_norm" else shape[1]
    w, b = torch.randn(c, device=dev, dtype=dt), torch.randn(c, device=dev, dtype=dt)
    xs = [torch.randn(*shape, device=dev, dtype=dt).requires_grad_(True) for _ in range(copies)]
    dy = torch.randn(*shape, device=dev, dtype=dt)
    t = torch.randn(shape[0], c, device=dev, dtype=dt) if "add" in kind else None
    silu = "silu" in kind
    if kind == "layer_norm":
        fused = lambda x: norms.layer_norm(x, w, b, eps)
        stock = lambda x: F.layer_norm(x, (c,), w, b, eps)
    else:
        fused = lambda x: norms.group_norm(x, groups, w, b, eps, silu=silu, channel_add=t)

        def stock(x):
            y = F.group_norm(x if t is None else x + t[:, :, None, None], groups, w, b, eps)
            return F.silu(y) if silu else y
    res = {"kind": kind, "shape": list(shape), "groups": groups, "input_copies": copies}
    # bytes: forward reads x (+ the [N, C] term) and writes y; backward reads x, dy (+ term) and writes dx
    fwd_bytes = 2 * xbytes
    bwd_bytes = 3 * xbytes
    for arm, fn in (("fused", fused), ("stock", stock)):
        def fwd():
            with torch.no_grad():
                for x in xs:
                    fn(x)

        def fwd_bwd():
            for x in xs:
                torch.autograd.grad(fn(x), x, dy)
        tf = timed(fwd, reps) / copies
        tb = timed(fwd_bwd, reps) / copies - tf
        res[arm] = {"fwd_us": round(tf, 2), "bwd_us": round(tb, 2), "fwd_GBps": round(fwd_bytes / tf / 1e3, 1),
                    "bwd_GBps": round(bwd_bytes / tb / 1e3, 1)}
    res["fwd_speedup"] = round(res["stock"]["fwd_us"] / res["fused"]["fwd_us"], 2)
    res["bwd_speedup"] = round(res["stock"]["bwd_us"] / res["fused"]["bwd_us"], 2)
    del xs
    return res


def micro_step_ab(norms, name, steps, rounds):
    """The graph-replayed micro-step of bench.py with and without the fused norms, arms alternated."""
    import pairwise_sample_optimization_b200 as pso
    L = pso._lib.lib()
    dev = torch.device("cuda", 0)
    args = bench.parse_args(["--config", name, "--no-cpu-baseline", "--no-eager-baseline"])
    arms = {}
    for arm in ("stock", "fused"):
        a = bench.B200Arm(args, name, dev, 0, 1, L)
        if arm == "fused":
            counts = norms.install_fused_norms(a.unet)
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        a.micro(a.d)  # one eager micro-step: its peak over what the arm holds at rest
        torch.cuda.synchronize()
        peak = torch.cuda.max_memory_allocated() - base
        a.bucket.zero_()
        a.capture()
        arms[arm] = {"arm": a, "peak_step_bytes": peak, "ms": []}
    loss = {}
    for _ in range(rounds):
        for arm in ("stock", "fused"):
            a = arms[arm]["arm"]
            for i in range(2):
                a.step(i)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for i in range(steps):
                a.graph.replay()
            e1.record()
            torch.cuda.synchronize()
            arms[arm]["ms"].append(e0.elapsed_time(e1) / steps)
            loss[arm] = float(a.static_loss.item())
            a.bucket.zero_()
    out = {"config": name, "pairs": args.pairs, "norm_modules_patched": counts, "steps_per_round": steps, "rounds": rounds}
    for arm in ("stock", "fused"):
        out[arm] = {"ms_per_micro_step_rounds": [round(v, 3) for v in arms[arm]["ms"]],
                    "ms_per_micro_step_median": round(statistics.median(arms[arm]["ms"]), 3),
                    "eager_micro_step_peak_GB": round(arms[arm]["peak_step_bytes"] / 1e9, 3), "loss": loss[arm]}
        arms[arm]["arm"].close()
    out["speedup"] = round(out["stock"]["ms_per_micro_step_median"] / out["fused"]["ms_per_micro_step_median"], 4)
    del arms
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", default="dmd128,turbo64")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--no-micro-step", action="store_true")
    ap.add_argument("--json", default=None, help="also write every result to this file")
    args = ap.parse_args()
    from pairwise_sample_optimization_b200 import norms
    report = {"card": card(), "shapes": [], "micro_step": []}
    print(json.dumps(report["card"]), flush=True)
    configs = args.configs.split(",")
    keys = {}
    for name in configs:
        for key, n in norm_shapes(bench.CONFIGS[name]["latent_hw"], 8).items():
            keys.setdefault(key, {})[name] = n
    for key, per_config in sorted(keys.items(), key=lambda kv: (kv[0][0], kv[0][1])):
        r = per_shape(norms, key, args.reps)
        r["launches_per_forward"] = per_config
        report["shapes"].append(r)
        print(json.dumps(r), flush=True)
    if not args.no_micro_step:
        for name in configs:
            r = micro_step_ab(norms, name, args.steps, args.rounds)
            report["micro_step"].append(r)
            print(json.dumps(r), flush=True)
    report["card_after"] = card()
    if args.json:
        with open(args.json, "w") as f:
            json.dump(report, f, indent=1)


if __name__ == "__main__":
    main()

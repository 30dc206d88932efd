#!/usr/bin/env python
"""Kernel-time breakdown of one eager micro-step of bench.py's workload (torch.profiler / CUPTI)."""
import os, sys, collections
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench
import pairwise_sample_optimization_b200 as pso
from fixtures import micro_step, sdxl_unet
from pairwise_sample_optimization_b200 import lora
from torch.profiler import profile, ProfilerActivity

import argparse
ap = argparse.ArgumentParser()
ap.add_argument("--config", default="dmd128", choices=sorted(bench.CONFIGS))
ap.add_argument("--pairs", type=int, default=4)
ap.add_argument("--top", type=int, default=40)
ap.add_argument("--grad-checkpointing", action="store_true")
ap.add_argument("--no-fused-geglu", action="store_true")
ap.add_argument("--fused-norms", action="store_true", help="LayerNorm / GroupNorm (+ SiLU) on the fused kernels (norms.install_fused_norms)")
args = ap.parse_args()
conf = bench.CONFIGS[args.config]
dev = torch.device("cuda", 0)
torch.manual_seed(1234)
cfg = sdxl_unet.sdxl_config()
with torch.device(dev):
    unet = sdxl_unet.UNet2DConditionModel(cfg)
unet = unet.to(torch.bfloat16).requires_grad_(False)
wrapped = lora.add_adapter(unet, lora.LoraConfig(r=conf["rank"], lora_alpha=conf["rank"]))
for m in wrapped:
    torch.nn.init.normal_(m.lora_B["default"].weight, std=0.01)
unet.set_attn_processor(lora.PSOAttnProcessor2_0()); unet.train()
if args.grad_checkpointing:
    unet.enable_gradient_checkpointing()
if not args.no_fused_geglu:
    from pairwise_sample_optimization_b200 import feed_forward
    feed_forward.install_fused_geglu(unet)
if args.fused_norms:
    from pairwise_sample_optimization_b200 import norms
    norms.install_fused_norms(unet)
bucket = lora.LoRAGradBucket(lora.lora_parameters(unet))
sched = bench.turbo_scheduler() if conf["kind"] == "turbo" else bench.dmd_scheduler()
host = micro_step.batched_view(micro_step.synth_batch(args.pairs, conf["latent_hw"], 2048, 1280, 100, getattr(sched, "sigmas", None),
                                                      dtype=torch.bfloat16, kind=conf["kind"]))
d = {k: v.to(dev) for k, v in host.items()}
step = lambda: micro_step.product_micro_step_batched(pso, lora, unet, d, sched, loss_scale=1 / 6, kind=conf["kind"])
for _ in range(3):
    step()
torch.cuda.synchronize()
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    step()
    torch.cuda.synchronize()
tot = collections.Counter(); cnt = collections.Counter()
for e in prof.events():
    if e.device_type.name == "CUDA":
        name = e.name.split("<")[0][:70]
        tot[name] += e.device_time if hasattr(e, "device_time") else e.cuda_time
        cnt[name] += 1
total = sum(tot.values())
print(f"total kernel time {total / 1e3:.1f} ms over {sum(cnt.values())} launches")
for name, t in tot.most_common(args.top):
    print(f"{t / 1e3:8.2f} ms {100 * t / total:5.1f}%  x{cnt[name]:5d}  avg {t / cnt[name]:7.1f} us  {name}")

# ---- which ATen operators the time belongs to (CPU-side op -> device time of the kernels it launched)
with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA], record_shapes=True) as prof2:
    step()
    torch.cuda.synchronize()
print(prof2.key_averages(group_by_input_shape=True).table(sort_by="self_device_time_total", row_limit=args.top,
                                                          max_name_column_width=40, max_shapes_column_width=70))

# ---- who launches the non-vectorised `elementwise_kernel`s (strided copies, broadcasts): op, shapes, enclosing ops
agg = collections.defaultdict(lambda: [0.0, 0])
for e in prof2.events():
    for k in getattr(e, "kernels", []) or []:
        if "elementwise_kernel" in k.name and "vectorized" not in k.name:
            chain, p = [], e.cpu_parent
            while p is not None and len(chain) < 3:
                chain.append(p.name)
                p = p.cpu_parent
            key = (e.name, str(e.input_shapes)[:90], " < ".join(chain))
            agg[key][0] += k.duration
            agg[key][1] += 1
print("\nnon-vectorised elementwise kernels by launching operator:")
for key, (t, n) in sorted(agg.items(), key=lambda kv: -kv[1][0])[:30]:
    print(f"{t / 1e3:8.2f} ms x{n:4d}  {key[0]}  {key[1]}  <- {key[2]}")

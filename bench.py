#!/usr/bin/env python
"""bench.py -- PSO train pairs/sec on synthetic SDXL-shaped data (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--pairs B] [--dump-outputs DIR]

Workload (config.workload): the configuration BASELINE.json's metric is quoted on ("SDXL 128x128 latents") = configs[2]'s
per-GPU slice: SDXL-DMD2 online PSO, LoRA rank 64, 1024x1024 (128x128 latents), bf16 (`--config dmd128`, default); configs[1]
(SDXL-Turbo, rank 8, 64x64 latents) is `--config turbo64`.  Both run on a random-init SDXL-ARCHITECTURE UNet
(fixtures/sdxl_unet.py: 2.57 B parameters, 70 transformer blocks, 560 LoRA-wrapped attention projections; diffusers is not
installed here).  A "step" is one training micro-step over B pairs, written as the reference writes it
(train_online_pso_sdxl_dmd2.py:773-864 / train_online_pso_sdxl_turbo.py:771-861):

    2 UNet forwards with grad (policy) + 2 adapter-disabled forwards without (frozen reference); activations stay resident
        (gradient checkpointing, the reference's memory workaround at :358, is `--grad-checkpointing`: same gradients, +28 % time)
    fused PSO loss+grad kernel  (replaces 4 x turbo_step_with_logprob + the inline loss + its backward)
    backward through the UNet   (LoRA dX / dA / dB on the tcgen05 GEMM path, accumulated into ONE flat fp32 buffer)
    every `accum` = GA x T = 6 steps: exchange of the flat LoRA gradient (N > 1: one multimem kernel of ours over the NVLink
    multicast mapping, fused with the gradient-norm pass; `--exchange nccl` = ncclAllReduce), then clip + AdamW +
    zero_grad + operand refresh fused over the flat buffers (2 launches)

The 560 projections (forward + backward), the loss and the feed-forward's gated GELU run on this repo's sm_100a kernels;
convolutions, norms, the feed-forward GEMMs and the attention core are stock torch kernels (outside the PSO hot path, SURVEY.md section 8).  One rank per GPU, pairs sharded
over ranks (weak scaling); the only collective is the LoRA-gradient all-reduce.

Numbers on the JSON line:
  value / ms_per_step : exactly K steps, inputs resident in HBM, CUDA events, max over ranks.
  e2e                 : the same K steps with the step's inputs copied from pinned host memory and the loss read back,
                        every step, inside the timed region.
  roofline            : the dominant kernel of OURS in this step -- the tensor-bound main passes of the LoRA-wrapped
                        projections (lora_gemm2_kernel, CTA pairs) -- one CUDA-event pair around EVERY launch in a separate
                        instrumented pass; achieved = 2 M N (K + r) flops per launch / launch time; peak = sustained bf16 TF/s.
  lora_skinny_launches: the rank-r side launches (t, u, dA, dB: HBM / latency bound) of the same pass, as GB/s of their
                        algorithmic bytes against the measured HBM copy bandwidth.
  loss_kernel_roofline / lora_gemm_large : the two kernel-level figures of BASELINE config 5 (fused loss+grad kernel at 256
                        pairs x 128x128 latents against the HBM roofline; the fused base+LoRA GEMM at M = 18944).
  sampler_kernel_roofline : step_logprob_kernel (sampling mode) at 256 x 4x128x128 bf16 against the HBM roofline.
  gpu_eager_baseline  : the reference's flow on THIS GPU with stock torch kernels -- the same fixture and batch, stock
                        nn.Linear + the peft-style LoRA module (3 cuBLAS GEMMs + scale + add per projection), 4 separate UNet
                        forwards, 4 step-with-logprob calls, inline loss, autograd -- eager and (where it captures) replayed
                        from a CUDA graph: the honest "reference on this box" figure (SURVEY.md section 8d, BASELINE.md section 3).
  lora_projection_vs_cublas : one LoRA-wrapped projection forward + backward, this library against 3 x cuBLAS + scale + add
                        under autograd, at the three in-step shapes of the workload.
  gate / grad_norm    : fraction of (pair, branch) clamp gates that were open in the timed step and the gradient norm of the
                        last optimizer boundary (a closed gate would make the backward vacuous).
  exchange_check      : N > 1: the gradient exchange of this run against ncclAllReduce(AVG) on a copy, outside the timed region.
  turbo64             : a short run of BASELINE configs[1] appended after the main timing (value, ms_per_step, roofline).
  cpu_baseline        : the oracle port of the reference's PyTorch path (fp32, same UNet architecture) on this box's host
                        cores, one micro-step of ONE pair (bounded sample), N = 1 / rank 0 only.
`--dump-outputs DIR` writes what the last timed step left for its caller as DIR/<name>.npy (see dump_outputs), so that two
builds can be compared output for output on the same seeded inputs.
`--impl reference` times that oracle port as the reference arm (the reference is Python that needs diffusers / peft /
accelerate and /root/reference; none exist on the GPU box -- DESIGN.md).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "pso_train_pairs_per_sec"
UNIT = "pairs/s"
ACCUM = 6  # gradient_accumulation_steps (2) x trained timesteps (3): turbo trainer :232, dmd2 trainer :236
DUMP_SAMPLE = 1 << 21  # --dump-outputs: at most 4 x 8 MB of float32 from the flat LoRA buffers
_COMMON = ("online PSO micro-step (2 policy + 2 frozen-reference UNet forwards, fused PSO loss+grad, backward), random-init "
           "SDXL-architecture UNet (2.57 B params, 560 LoRA projections), bf16, optimizer step every 6 micro-steps")
# BASELINE.json's metric is quoted on SDXL 128x128 latents = configs[2] (SDXL-DMD2, rank 64, 1024 px): the default.
# configs[1] (SDXL-Turbo, rank 8, 64x64 latents, the reference's 512-px recipe) is `--config turbo64`.
CONFIGS = {
    "dmd128": {"kind": "dmd", "latent_hw": 128, "rank": 64,
               "workload": "BASELINE configs[2] per-GPU slice: SDXL-DMD2 " + _COMMON + ", LoRA rank 64, 128x128 latents (1024 px)"},
    "turbo64": {"kind": "turbo", "latent_hw": 64, "rank": 8,
                "workload": "BASELINE configs[1]: SDXL-Turbo " + _COMMON + ", LoRA rank 8, 64x64 latents (512 px)"},
    # configs[3]: train_pso_sdxl_turbo_dreambooth.py:1720-1964; a "pair" = one (win, lose) image pair = 2 rows of the 2b-row batch
    "dreambooth64": {"kind": "dreambooth", "latent_hw": 64, "rank": 4,
                     "workload": "BASELINE configs[3]: SDXL-Turbo DreamBooth-style PSO micro-step (1 policy + 1 frozen-reference "
                                 "UNet forward of 2b rows, fused DreamBooth-PSO loss+grad [pso, beta 5, neg_defactor 0.1, prior 0.5], "
                                 "backward), random-init SDXL-architecture UNet, bf16, LoRA rank 4, 64x64 latents (512 px), "
                                 "optimizer step every 4 micro-steps"},
}


# ----------------------------------------------------------------------------------------------- utilities
def dist_env():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))


class ClockSampler:
    """Samples SM clock and throttle reasons during the timed region (NVML, falls back to nvidia-smi)."""

    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index: int):
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _poll(self):
        while not self._stop.is_set():
            try:
                if self.nv is not None:
                    self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                    mask = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                    for bit, name in self.REASONS.items():
                        if mask & bit:
                            self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.02)

    def __enter__(self):
        self._thread = threading.Thread(target=self._poll, daemon=True)
        self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        self._thread.join()

    def summary(self):
        if not self.samples:
            try:
                import subprocess
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", "--query-gpu=clocks.sm,clocks.max.sm",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=10)
                sm, mx = (int(v) for v in out.stdout.strip().split(","))
                return {"sm_mhz": sm, "sm_max_mhz": mx, "reasons": sorted(self.reasons), "note": "sampled after the timed region"}
            except Exception:
                return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": []}
        return {"sm_mhz": int(statistics.median(self.samples)), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"hbm": float(p["hbm_gbs"]), "tf_burst": float(p["bf16_tflops"]),
                "tf_sustained": float(p.get("bf16_tflops_sustained", p["bf16_tflops"])),
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm": 6650.0, "tf_burst": 1590.0, "tf_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


def dmd_scheduler():
    """SDXL alphas_cumprod (scaled_linear betas; restated, see oracle/schedules.py): all the DMD2 / LCM step reads."""
    import types
    betas = torch.linspace(0.00085 ** 0.5, 0.012 ** 0.5, 1000, dtype=torch.float32) ** 2
    return types.SimpleNamespace(alphas_cumprod=torch.cumprod(1.0 - betas, dim=0))


def turbo_scheduler():
    """SDXL-Turbo EulerAncestral schedule, 4 trailing steps (restated; see oracle/schedules.py for the anchored copy)."""
    import types
    betas = torch.linspace(0.00085 ** 0.5, 0.012 ** 0.5, 1000, dtype=torch.float32) ** 2
    ac = torch.cumprod(1.0 - betas, dim=0)
    ts = torch.tensor([999, 749, 499, 249])
    sig = ((1 - ac) / ac) ** 0.5
    return types.SimpleNamespace(timesteps=ts.float(), sigmas=torch.cat([sig[ts], torch.zeros(1)]).float())


def graph_timed(fn, reps, per_graph=2):
    """Mean device time (ms) of one ``fn()`` call: calls captured in a CUDA graph, one event pair per replay."""
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=side):
        for _ in range(per_graph):
            fn()
    for _ in range(3):
        graph.replay()
    torch.cuda.synchronize()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in evs:
        a.record()
        graph.replay()
        b.record()
    torch.cuda.synchronize()
    return statistics.mean(a.elapsed_time(b) for a, b in evs) / per_graph


# ----------------------------------------------------------------------------------------------- kernel-level figures
def loss_kernel_roofline(pso, dev, peaks):
    """Fused loss+grad kernel alone at the top of the config-5 sweep: 256 pairs of 4x128x128 bf16 latents (DMD2 shapes);
    inputs (336 MB) exceed L2.  Algorithmic bytes = 10 N sizeof(bf16) per pair (SURVEY.md section 8d)."""
    import types
    B, n = 256, 4 * 128 * 128
    g = torch.Generator(device=dev).manual_seed(7)
    mk = lambda: torch.randn(B, 4, 128, 128, device=dev, generator=g).bfloat16()
    x0, x1, r0, r1, n0, n1 = mk(), mk(), mk(), mk(), mk(), mk()
    p0 = (r0.float() + 0.02 * torch.randn_like(r0, dtype=torch.float32)).bfloat16()
    p1 = (r1.float() + 0.02 * torch.randn_like(r1, dtype=torch.float32)).bfloat16()
    ts = torch.tensor([999, 749, 499], device=dev)[torch.randint(0, 3, (B,), device=dev)]
    h = torch.tensor([[-1.0, 1.0]], device=dev).repeat(B, 1)
    betas = torch.linspace(0.00085 ** 0.5, 0.012 ** 0.5, 1000, dtype=torch.float32) ** 2
    sched = types.SimpleNamespace(alphas_cumprod=torch.cumprod(1.0 - betas, dim=0).to(dev))

    def call():
        with torch.no_grad():
            pso.pso_pair_loss(p0, p1, r0, r1, x0, x1, n0, n1, ts, ts, h, scheduler=sched, kind="dmd", step_ratio=250)
    ms = graph_timed(call, 20, per_graph=1)
    alg = 10 * n * 2 * B
    ach = alg / (ms * 1e-3) / 1e9
    traffic, traffic_src = ncu_traffic("pair_loss_grad_tmem_kernel@256x4x128x128_bf16")
    return {"kernel": "pair_loss_grad_tmem_kernel<bf16,bf16,ref>", "bound": "hbm", "achieved": round(ach, 1), "peak": peaks["hbm"],
            "unit": "GB/s", "frac": round(ach / peaks["hbm"], 4), "traffic": traffic, "traffic_source": traffic_src,
            "workload": "256 pairs x 4x128x128 bf16 (BASELINE config 5 top of sweep)", "algorithmic_bytes_per_launch": alg,
            "avg_launch_us": round(ms * 1e3, 2), "peak_source": peaks["source"]}


def lora_gemm_large(dev, peaks):
    """Fused base+LoRA projection y = x W^T + b + t B^T (one launch) at M = 18944 (148 row tiles), K = N = 1280, r = 64."""
    from pairwise_sample_optimization_b200 import gemm
    M, K, N, r = 18944, 1280, 1280, 64
    g = torch.Generator(device=dev).manual_seed(3)
    rn = lambda *s, sc=1.0: (torch.randn(*s, device=dev, generator=g) * sc).bfloat16()
    x, w, b, A, Bm = rn(M, K), rn(N, K, sc=K ** -0.5), rn(N), rn(r, K, sc=1 / r), rn(N, r, sc=0.05)
    T, _ = gemm.lora_gemm(x, A)
    out = torch.empty(M, N, device=dev, dtype=torch.bfloat16)
    ms = graph_timed(lambda: gemm.lora_gemm(x, w, T, Bm, bias=b, out=out), 20)
    fl = 2.0 * M * N * (K + r)
    ach = fl / (ms * 1e-3) / 1e12
    return {"kernel": "lora_gemm_kernel (x W^T + b + t B^T)", "bound": "tensor", "achieved": round(ach, 1),
            "peak": peaks["tf_burst"], "unit": "TFLOP/s", "frac": round(ach / peaks["tf_burst"], 4),
            "shape": {"M": M, "K": K, "N": N, "r": r}, "avg_launch_us": round(ms * 1e3, 2), "peak_source": peaks["source"]}


# ----------------------------------------------------------------------------------------------- b200 arm
def ncu_traffic(key):
    """(bytes per launch, source) of a committed `ncu --set full` capture (profiles/ncu_traffic.json), else (None, None)."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        with open(path) as f:
            e = json.load(f).get(key)
        return (e["bytes"], e["source"]) if e else (None, None)
    except Exception:
        return None, None


def config_block(args, name):
    """The `config` object of the JSON line: names the WORKLOAD only, so that both arms print the same object."""
    conf = CONFIGS[name]
    out = {"workload": conf["workload"] if not args.tiny else "TINY fixture (debug run, not the benchmark)", "name": name,
           "pairs_per_gpu_per_step": args.pairs, "latent_shape": [4, conf["latent_hw"], conf["latent_hw"]],
           "lora_rank": conf["rank"]}
    out.update({"loss_type": "pso", "beta_pso": 5.0, "neg_defactor": 0.1, "prior_loss_weight": 0.5, "accum": 4}
               if conf["kind"] == "dreambooth" else {"beta": 50.0, "eps": 0.1, "accum": ACCUM})
    return out


def dreambooth_scheduler():
    """EulerDiscreteScheduler as constructed (no set_timesteps): timesteps 999..0, sigmas descending + [0] (restated; the
    anchored copy is oracle/schedules.py::dreambooth_scheduler; dreambooth trainer :1235-1237, :1675-1685)."""
    import types
    betas = torch.linspace(0.00085 ** 0.5, 0.012 ** 0.5, 1000, dtype=torch.float64) ** 2
    ac = torch.cumprod(1.0 - betas, dim=0)
    sig = (((1 - ac) / ac) ** 0.5).flip(0)
    return types.SimpleNamespace(timesteps=torch.arange(999, -1, -1, dtype=torch.float32),
                                 sigmas=torch.cat([sig, torch.zeros(1, dtype=torch.float64)]).float())


def make_scheduler(kind, dev=None):
    sched = turbo_scheduler() if kind == "turbo" else dmd_scheduler()
    if dev is not None:
        for k, v in list(vars(sched).items()):
            setattr(sched, k, v.to(dev))
    return sched


class B200Arm:
    """One workload configuration on this repo's kernels: model, flat optimizer, static device batch, captured micro-step."""

    def __init__(self, args, name, dev, rank, world, L):
        import pairwise_sample_optimization_b200 as pso
        from fixtures import micro_step, sdxl_unet
        from pairwise_sample_optimization_b200 import lora
        self.args, self.name, self.dev, self.rank, self.world, self.L = args, name, dev, rank, world, L
        self.pso, self.lora, self.micro_step = pso, lora, micro_step
        conf = CONFIGS[name]
        self.kind, self.hw, self.r = conf["kind"], conf["latent_hw"], conf["rank"]
        self.B = args.pairs
        # ---- model: random-init SDXL-architecture UNet in bf16, LoRA on to_q/to_k/to_v/to_out.0
        torch.manual_seed(1234)  # same base weights on every rank (as a checkpoint would give)
        cfg = sdxl_unet.tiny_config() if args.tiny else sdxl_unet.sdxl_config()
        with torch.device(dev):
            unet = sdxl_unet.UNet2DConditionModel(cfg)
        unet = unet.to(torch.bfloat16).requires_grad_(False)
        wrapped = lora.add_adapter(unet, lora.LoraConfig(r=self.r, lora_alpha=self.r))
        for m in wrapped:  # the reference starts from B = 0; use a small non-zero B so every adapter GEMM does real work
            torch.nn.init.normal_(m.lora_B["default"].weight, std=0.01)
        unet.set_attn_processor(lora.PSOAttnProcessor2_0())
        if args.fuse_projections:  # q / k / v (k / v) of every attention stacked into one launch per direction
            lora.fuse_attention_projections(unet)
            if args.kv_bank:  # the k / v projections of all 70 cross-attention layers (prompt embeddings only): one launch per shape
                lora.fuse_cross_attention_kv(unet)
        if args.fused_geglu:  # the feed-forward's gated GELU on one fused kernel each way (outside SURVEY section 8's rows)
            from pairwise_sample_optimization_b200 import feed_forward
            feed_forward.install_fused_geglu(unet)
        lora.set_wgrad_stream(args.wgrad_stream)
        lora.set_in_launch_dependencies(not args.no_inlaunch_deps)
        lora.set_programmatic_launch(args.programmatic_launch)
        # --deterministic (default): the same arguments compute the same outputs on every run, which is what --dump-outputs
        # compares -- dA / dB reductions not split over CTAs (one accumulation per element and launch) and the stock torch
        # kernels of the step on their deterministic algorithms, for the lifetime of this arm (close() restores the defaults)
        lora.set_deterministic_wgrad(args.deterministic)
        torch.use_deterministic_algorithms(args.deterministic)
        unet.train()
        if args.grad_checkpointing:
            unet.enable_gradient_checkpointing()  # turbo trainer :358
        self.unet, self.cfg = unet, cfg
        # parameters, gradients and Adam moments of all 1120 adapter matrices live in four flat fp32 buffers: the optimizer
        # boundary is one exchange + two launches (clip + AdamW + zero_grad + 16-bit operand refresh).  Data-parallel exchange:
        # one kernel of ours per rank over the NVLink multicast mapping (in-switch reduction fused with the norm pass of
        # clip_grad_norm_); `--exchange nccl` (or a group without multicast support) = one NCCL all-reduce
        opt_kw = dict(lr=1e-5, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-4, max_grad_norm=1.0)
        self.opt, self.exchange_kind = None, "none (1 GPU)"
        if world > 1 and args.exchange == "multimem":
            try:
                self.opt = lora.FusedLoRAOptimizer(unet, exchange=lora.SymmetricGradExchange(), **opt_kw)
                self.exchange_kind = "multimem.ld_reduce/st kernel fused with the gradient-norm pass (NVLink SHARP), no NCCL call"
            except Exception as e:  # no NVSwitch multicast on this box: same on every rank
                print(f"[bench] symmetric-memory exchange unavailable ({type(e).__name__}: {e}); using NCCL", file=sys.stderr)
        if self.opt is None:
            self.opt = lora.FusedLoRAOptimizer(unet, **opt_kw)
            if world > 1:
                self.exchange_kind = "one NCCL all-reduce of the flat gradient"
        self.bucket = self.opt.bucket
        self.accum = 4 if self.kind == "dreambooth" else ACCUM  # pso_dog.sh: gradient_accumulation_steps 4
        pooled = cfg.projection_class_embeddings_input_dim - 6 * cfg.addition_time_embed_dim
        if self.kind == "dreambooth":
            self.sched = dreambooth_scheduler()
            host = micro_step.synth_dreambooth_batch(self.B, self.hw, cfg.cross_attention_dim, pooled, 100 + rank, self.sched,
                                                     dtype=torch.bfloat16)
        else:
            self.sched = make_scheduler(self.kind)
            host = micro_step.synth_batch(self.B, self.hw, cfg.cross_attention_dim, pooled, 100 + rank,
                                          getattr(self.sched, "sigmas", None), dtype=torch.bfloat16, kind=self.kind)
            if not args.separate_forwards:
                host = micro_step.batched_view(host)
        self.host = {k: v.pin_memory() for k, v in host.items()}
        self.d = {k: v.to(dev) for k, v in self.host.items()}
        self.fwd_bwd = micro_step.product_micro_step if args.separate_forwards else micro_step.product_micro_step_batched
        self.ref_stream = torch.cuda.Stream() if (args.overlap_reference and not args.separate_forwards) else None
        self.graph = self.static_loss = self.side = None
        self.launches_per_micro = 0
        self.one_step = None

    # ---- one micro-step (turbo trainer :771-861 / dmd2 trainer :773-864)
    def micro(self, batch, overlap=True, **extra):
        kw = {"ref_stream": self.ref_stream} if (self.ref_stream is not None and overlap) else {}
        if self.kind == "dreambooth":  # dreambooth trainer :1812-1953 (pso_dog.sh: beta_pso 5, prior_loss_weight 0.5)
            return self.micro_step.product_dreambooth_micro_step(self.pso, self.lora, self.unet, batch, loss_type="pso",
                                                                 beta_pso=5.0, neg_defactor=0.1, prior_loss_weight=0.5,
                                                                 loss_scale=1.0 / self.accum, **kw, **extra)
        return self.fwd_bwd(self.pso, self.lora, self.unet, batch, self.sched, beta=50.0, eps=0.1, loss_scale=1.0 / ACCUM,
                            kind=self.kind, **kw, **extra)

    def optimizer_boundary(self, i):
        if (i + 1) % self.accum == 0:  # turbo trainer :858-861 (sync_gradients): exchange, clip, AdamW, zero_grad
            self.opt.all_reduce()
            self.opt.step()

    def capture(self):
        # warm up eagerly on a side stream (also fills every host-side cache), then capture ONE micro-step: forward(s),
        # fused loss+grad kernel, backward with in-place accumulation into the flat bucket.  Replays need no Python.
        self.side = torch.cuda.Stream()
        self.side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(self.side):
            for _ in range(3):
                self.micro(self.d)
        torch.cuda.current_stream().wait_stream(self.side)
        torch.cuda.synchronize()
        self.pso.check_status(self.dev)
        self.bucket.zero_()
        self.graph = torch.cuda.CUDAGraph()
        n0 = self.L.psob200_launch_count()
        with torch.cuda.graph(self.graph, stream=self.side):
            self.static_loss = self.micro(self.d)
        self.launches_per_micro = self.L.psob200_launch_count() - n0  # kernels of this library inside the captured micro-step
        self.bucket.zero_()

    def step(self, i):
        if self.graph is not None:
            self.graph.replay()  # the captured micro-step reads the static device batch `d`
            loss = self.static_loss
        else:
            loss = self.micro(self.d)
        self.optimizer_boundary(i)
        return loss

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, ms: float) -> float:
        if self.world > 1:
            import torch.distributed as dist
            t = torch.tensor([ms], device=self.dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return ms

    def timed(self, K, W):
        """Exactly K steps, inputs resident in HBM, CUDA events, max over ranks."""
        for i in range(W):
            self.step(i)
        self.optimizer_boundary(self.accum - 1)  # one untimed optimizer boundary: first exchange, kernels loaded
        self.pso.check_status(self.dev)
        self.bucket.zero_()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.barrier()
        launches0 = self.L.psob200_launch_count()
        with ClockSampler(self.dev.index) as clocks:
            marks = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]
            ev0.record()
            marks[0].record()
            for i in range(K):
                if self.args.profiler_range and i == K - 1:  # ncu --profile-from-start off: exactly the last timed step
                    torch.cuda.profiler.start()
                loss = self.step(i)
                if self.args.profiler_range and i == K - 1:
                    torch.cuda.synchronize()
                    torch.cuda.profiler.stop()
                marks[i + 1].record()
            ev1.record()
            self.barrier()
        self.last_loss = loss
        launches = self.L.psob200_launch_count() - launches0 + K * self.launches_per_micro
        per_step = [marks[i].elapsed_time(marks[i + 1]) for i in range(K)]
        ms_per_step = self.max_over_ranks(ev0.elapsed_time(ev1)) / K
        out = {"value": self.world * self.B / (ms_per_step * 1e-3), "ms_per_step": ms_per_step, "per_step": per_step,
               "launches": int(launches), "clocks": clocks.summary(), "loss": float(loss.item()) * self.accum}
        if K >= self.accum:  # at least one optimizer boundary inside the timed region: its (pre-clip) gradient norm
            out["grad_norm"] = float(self.opt.grad_norm.item())
        return out

    def dump_outputs(self, out_dir):
        """What the last timed step left for its caller, as float32 .npy files: the loss it returned, the gradient norm of
        the last optimizer boundary, and the four flat LoRA buffers (adapter parameters, accumulated gradient, both AdamW
        moments).  A buffer longer than DUMP_SAMPLE elements is stored at DUMP_SAMPLE positions drawn with a fixed seed."""
        import numpy as np
        os.makedirs(out_dir, exist_ok=True)
        bufs = {"lora_params": self.opt.flat_param, "lora_grad": self.bucket.flat, "adamw_exp_avg": self.opt.exp_avg,
                "adamw_exp_avg_sq": self.opt.exp_avg_sq}
        n = self.bucket.flat.numel()
        idx = None
        if n > DUMP_SAMPLE:
            idx = torch.randint(0, n, (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(0)).sort().values.to(self.dev)
        out = {"loss": self.last_loss.detach(), "grad_norm": self.opt.grad_norm}
        out.update({k: (v if idx is None else v[idx]) for k, v in bufs.items()})
        for k, v in out.items():
            np.save(os.path.join(out_dir, k + ".npy"), v.float().cpu().numpy())

    def e2e(self, K):
        """The same K steps with the step's inputs copied from pinned host memory and the loss read back, every step."""
        loss_pinned = torch.empty((), dtype=torch.float32).pin_memory()
        h2d_bytes = sum(v.numel() * v.element_size() for v in self.host.values())

        def e2e_step(i):
            for k, v in self.host.items():
                self.d[k].copy_(v, non_blocking=True)
            loss = self.step(i)
            loss_pinned.copy_(loss.detach(), non_blocking=True)
            torch.cuda.current_stream().synchronize()
            return float(loss_pinned)
        self.bucket.zero_()
        e2e_step(0)
        self.bucket.zero_()
        self.barrier()
        t0 = time.perf_counter()
        for i in range(K):
            e2e_step(i)
        torch.cuda.synchronize()
        e2e_ms = self.max_over_ranks((time.perf_counter() - t0) * 1e3)
        self.barrier()
        self.bucket.zero_()
        return {"value": round(self.world * self.B * K / (e2e_ms * 1e-3), 2), "unit": UNIT, "h2d_bytes_per_step": h2d_bytes,
                "d2h_bytes_per_step": 4, "ms_per_step": round(e2e_ms / K, 3)}

    def gate(self):
        """One eager micro-step (untimed) with the loss kernel's per-pair statistics: how many clamp gates were open."""
        if self.args.separate_forwards:
            return None
        self.bucket.zero_()
        loss1, stats = self.micro(self.d, return_stats=True)
        torch.cuda.synchronize()
        self.one_step = {"loss": float(loss1.item()) * self.accum, "grad": self.bucket.flat.clone()}  # for the eager-arm parity check
        self.bucket.zero_()
        if self.kind == "dreambooth" or stats is None:
            return None
        delta = stats[:, 4:6].double()  # log pi_theta - log pi_ref per branch
        h = self.d["human_prefer"].double()
        ratio = torch.exp(delta)
        open_ = ((ratio >= 1 - 0.1) & (ratio <= 1 + 0.1) & (h != 0)).double()
        return {"open_fraction": round(float(open_.mean().item()), 4), "pair_branches": int(open_.numel()),
                "max_abs_log_ratio": round(float(delta.abs().max().item()), 5),
                "note": "a (pair, branch) contributes gradient only while 1-eps <= pi_theta/pi_ref <= 1+eps (turbo :844-845)"}

    def instrumented(self, ms_per_step, peaks):
        """Roofline of the dominant kernel of ours: instrumented pass, ONE launch between each pair of events."""
        lora = self.lora
        self.bucket.zero_()
        sink = []
        lora.set_timing_sink(sink)
        if self.graph is None:
            self.micro(self.d, overlap=False)
        else:
            # captured like the timed step, with the event records as graph nodes: an eager pass is host-bound (the GPU idles
            # between a record and the launch behind it) and would charge host latency to the kernels
            self.side.wait_stream(torch.cuda.current_stream())
            inst_graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(inst_graph, stream=self.side):  # the stream the step was warmed up and captured on
                self.micro(self.d, overlap=False)  # one stream: a launch's interval must not include waiting for the other stream's CTAs
            for _ in range(2):
                inst_graph.replay()  # the events keep the timestamps of the last replay
        lora.set_timing_sink(None)
        torch.cuda.synchronize()
        is_main = lambda role: role.startswith("y =") or role.startswith("dx =") or role.startswith("qkv") or role.startswith("kv")
        agg = {True: [0.0, 0.0, 0.0, 0], False: [0.0, 0.0, 0.0, 0]}  # ms, flops, bytes, launches
        by_shape = {}
        for ev0, ev1, fl, by, role, shape in sink:
            ms = ev0.elapsed_time(ev1)
            a_ = agg[is_main(role)]
            a_[0] += ms; a_[1] += fl; a_[2] += by; a_[3] += 1
            t = by_shape.setdefault((role,) + tuple(shape), [0.0, 0, 0.0, 0.0])
            t[0] += ms; t[1] += 1; t[2] += fl; t[3] += by
        m_ms, m_fl, m_by, m_n = agg[True]
        s_ms, s_fl, s_by, s_n = agg[False]
        ach = m_fl / (m_ms * 1e-3) / 1e12 if m_ms > 0 else 0.0
        rows = [{"launch": k[0], "M": k[1], "K": k[2], "N": k[3], "r": k[4], "launches_per_step": v[1],
                 "avg_us": round(v[0] * 1e3 / v[1], 2), "ms_per_step": round(v[0], 2),
                 **({"tflops": round(v[2] / (v[0] * 1e-3) / 1e12, 1)} if is_main(k[0]) else
                    {"gbs": round(v[3] / (v[0] * 1e-3) / 1e9, 1)})}
                for k, v in sorted(by_shape.items(), key=lambda kv: -kv[1][0])]
        # per launch of the stacked q / k / v forward (the widest launch of the step); other launches: see profiles/r02_kernels.md
        traffic, traffic_src = (ncu_traffic("lora_gemm2_kernel@stacked_qkv_fwd_M8192_K1280_N3840_r64_bf16")
                                if self.name == "dmd128" and self.args.fuse_projections else (None, None))
        roofline = {"kernel": "lora_gemm2_kernel / lora_gemm_kernel main passes: y = x W^T + b + t B^T, dx = dy W + u A (tcgen05, "
                              "frozen weight + adapter in one pass; t / u as tiles of the same launch; q / k / v stacked) over the "
                              "560 LoRA-wrapped projections",
                    "bound": "tensor", "achieved": round(ach, 2), "peak": peaks["tf_sustained"], "unit": "TFLOP/s",
                    "frac": round(ach / peaks["tf_sustained"], 4), "traffic": traffic, "traffic_source": traffic_src,
                    "peak_source": peaks["source"] + ", sustained bf16 (kernel timed inside a long step)",
                    "launches_per_step": m_n, "avg_launch_us": round(m_ms * 1e3 / max(m_n, 1), 2),
                    "share_of_step": round(m_ms / ms_per_step, 4), "flops_per_step": m_fl,
                    "algorithmic_flops": "2 M N (K + r) per launch (r = 0 for the frozen-reference pass) + 2 M r K (2 M r N) for the "
                                         "in-launch t (u) tiles",
                    "by_launch": [r_ for r_ in rows if is_main(r_["launch"])],
                    "how": "one CUDA-event pair around EVERY launch (event records captured as graph nodes) in one extra replayed step on ONE "
                           "stream (in the timed step the frozen-reference forward shares the SMs from a second stream, which would "
                           "charge its CTAs' residency to these intervals); includes the graph-node gaps around each launch, so "
                           "slightly pessimistic"}
        s_ach = s_by / (s_ms * 1e-3) / 1e9 if s_ms > 0 else 0.0
        skinny = {"kernel": "lora_gemm_kernel rank-r side launches: dA += u^T x and dB += dy^T t of a projection (a stacked group) in "
                            "ONE split-K launch, u = s dy B alone where no dx is needed (cross-attention k / v); arithmetic "
                            "intensity <= 84 flop/B, SURVEY.md section 8d",
                  "bound": "hbm", "achieved": round(s_ach, 1), "peak": peaks["hbm"], "unit": "GB/s",
                  "frac": round(s_ach / peaks["hbm"], 4), "launches_per_step": s_n,
                  "avg_launch_us": round(s_ms * 1e3 / max(s_n, 1), 2), "share_of_step": round(s_ms / ms_per_step, 4),
                  "algorithmic_bytes": "operands read once + result written once per launch",
                  "by_launch": [r_ for r_ in rows if not is_main(r_["launch"])]}
        self.bucket.zero_()
        return roofline, skinny

    def exchange_check(self):
        """N > 1, outside the timed region: this run's gradient exchange (the multimem kernel, or NCCL with `--exchange nccl`)
        against ncclAllReduce(AVG) on a copy of the same per-rank data."""
        import torch.distributed as dist
        opt, dev = self.opt, self.dev
        flat = self.bucket.flat
        g = torch.Generator(device=dev).manual_seed(4242 + self.rank)
        src = torch.randn(flat.numel(), device=dev, generator=g) * (1.0 + self.rank)
        want = src.clone()
        dist.all_reduce(want, op=dist.ReduceOp.AVG)
        flat.copy_(src)
        del src
        opt.all_reduce()
        torch.cuda.synchronize()
        max_rel = float(((flat - want).abs().max() / want.abs().max()).item())
        bits = flat.view(torch.int32)
        hi, lo = bits.clone(), bits.clone()
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        bitwise = bool(torch.equal(hi, lo))
        del hi, lo
        want_norm = float(torch.linalg.vector_norm(want.double()).item())
        norm_rel = None
        if opt.exchange is not None:  # the sum of squares the fused kernel left for clip_grad_norm_, one part per rank
            ex = opt.exchange
            parts = ex.buffer[ex.n:ex.n + 2 * ex.world].view(torch.float64)
            norm_rel = abs(float(parts.sum().sqrt().item()) - want_norm) / want_norm
            ex.buffer[ex.n:].zero_()
            opt._parts_ready = False
        flat.zero_()
        self.barrier()
        worst = torch.tensor([max_rel, 0.0 if bitwise else 1.0, norm_rel or 0.0], device=dev, dtype=torch.float64)
        dist.all_reduce(worst, op=dist.ReduceOp.MAX)
        return {"against": "ncclAllReduce(AVG) of the same per-rank gradients (seeded N(0,(1+rank)^2)), outside the timed region",
                "exchange": self.exchange_kind, "elements": int(flat.numel()), "max_rel_err": float(worst[0].item()),
                "bitwise_equal_across_ranks": bool(worst[1].item() == 0.0),
                "norm_rel_err": (float(worst[2].item()) if norm_rel is not None else None)}

    def close(self):
        self.lora.set_wgrad_stream(False)
        self.lora.set_deterministic_wgrad(False)
        torch.use_deterministic_algorithms(False)
        self.graph = self.static_loss = None
        self.unet = self.opt = self.bucket = self.d = self.host = None
        import gc
        gc.collect()
        torch.cuda.empty_cache()


def lora_layers_in_module_order(unet):
    from pairwise_sample_optimization_b200 import lora
    return lora.lora_layers(unet)


def flat_order(arm):
    """For every LoRA layer in module order: (offset of A, offset of B) inside the arm's flat gradient buffer."""
    off = {id(p): o for p, o in zip(arm.bucket.params, arm.bucket.offsets)}
    return [(off[id(m.lora_A["default"].weight)], off[id(m.lora_B["default"].weight)]) for m in lora_layers_in_module_order(arm.unet)]


def sampler_kernel_roofline(dev, peaks):
    """step_logprob_kernel in sampling mode (x' = mu + s noise, log-prob, next scaled UNet input) alone: 256 samples of
    4x128x128 bf16, Euler-ancestral schedule.  Algorithmic bytes per sample = 3 N read (prediction, latent, noise) + 2 N written
    (next latent, next scaled input) (SURVEY.md section 8d)."""
    from pairwise_sample_optimization_b200 import _lib, runtime, step_ops
    B, n = 256, 4 * 128 * 128
    g = torch.Generator(device=dev).manual_seed(11)
    mk = lambda: torch.randn(B, 4, 128, 128, device=dev, generator=g).bfloat16()
    pred, x, noise = mk(), mk(), mk()
    ts = torch.tensor([999, 749, 499], device=dev)[torch.randint(0, 3, (B,), device=dev)]
    sched = runtime.turbo_schedule(make_scheduler("turbo", dev), dev, _lib.ts_dtype_code(ts))
    ms = graph_timed(lambda: step_ops.step_forward(sched, pred, x, ts, noise=noise, want_scaled_next=True), 20, per_graph=1)
    alg = 5 * n * 2 * B
    ach = alg / (ms * 1e-3) / 1e9
    traffic, src = ncu_traffic("step_logprob_kernel@256x4x128x128_bf16_sampling")
    return {"kernel": "step_logprob_kernel<bf16> sampling mode + fused next-input scaling", "bound": "hbm", "achieved": round(ach, 1),
            "peak": peaks["hbm"], "unit": "GB/s", "frac": round(ach / peaks["hbm"], 4), "traffic": traffic, "traffic_source": src,
            "workload": "256 samples x 4x128x128 bf16", "algorithmic_bytes_per_launch": alg,
            "avg_launch_us": round(ms * 1e3, 2), "peak_source": peaks["source"]}


def lora_projection_vs_cublas(dev, shapes, r):
    """One LoRA-wrapped projection, forward + backward (dX, dA, dB), through this library's public module against the stock
    lowering (F.linear x 3 + scale + add under autograd = what peft's lora.Linear runs on cuBLAS); CUDA events around graph replays."""
    from pairwise_sample_optimization_b200 import lora
    g = torch.Generator(device=dev).manual_seed(5)
    rn = lambda *s, sc=1.0: (torch.randn(*s, device=dev, generator=g) * sc).bfloat16()
    rows = []
    for (M, K, N) in shapes:
        x, dy = rn(M, K), rn(M, N)
        lay = lora.LoRALinear(torch.nn.Linear(K, N, bias=True, device=dev, dtype=torch.bfloat16), r, r)
        with torch.no_grad():
            lay.lora_B["default"].weight.normal_(std=0.02)
        w, b = lay.base_layer.weight, lay.base_layer.bias
        xg = x.clone().requires_grad_(True)
        xa = x.clone().requires_grad_(True)
        Ap = lay.lora_A["default"].weight.detach().bfloat16().clone().requires_grad_(True)
        Bp = lay.lora_B["default"].weight.detach().bfloat16().clone().requires_grad_(True)

        def ours():
            lay(xg).backward(dy)

        def stock():
            F = torch.nn.functional
            (F.linear(xa, w, b) + F.linear(F.linear(xa, Ap), Bp) * 1.0).backward(dy)
        t_o, t_s = graph_timed(ours, 10) * 1e3, graph_timed(stock, 10) * 1e3
        rows.append({"M": M, "K": K, "N": N, "r": r, "ours_fwd_bwd_us": round(t_o, 1), "cublas_fwd_bwd_us": round(t_s, 1),
                     "speedup": round(t_s / t_o, 3)})
    return rows


def gpu_eager_baseline(args, name, dev, host, reps=4, same_weights=None):
    """The reference's micro-step on THIS GPU with stock torch kernels: same architecture, same base weights (seed), same batch;
    stock nn.Linear + the peft-style LoRA module (oracle/lora.py: 3 cuBLAS GEMMs + scale + add), 4 separate forwards, the four
    step-with-logprob calls + inline loss restated in oracle/, autograd backward.  oracle/ is checker code: it is executed here
    only as a reported BASELINE, never on the product path.  bf16 weights AND bf16 adapters, activations resident (no gradient
    checkpointing): both more favourable to the baseline than the reference's shipped recipe."""
    from fixtures import micro_step, sdxl_unet
    from oracle import lora as olora, losses as olosses
    conf = CONFIGS[name]
    kind, r = conf["kind"], conf["rank"]
    torch.manual_seed(1234)
    cfg = sdxl_unet.tiny_config() if args.tiny else sdxl_unet.sdxl_config()
    with torch.device(dev):
        unet = sdxl_unet.UNet2DConditionModel(cfg)
    unet = unet.to(torch.bfloat16).requires_grad_(False)
    wrapped = olora.oracle_add_adapter(unet, r, r)
    for m in wrapped:
        torch.nn.init.normal_(m.lora_B["default"].weight, std=0.01)
        m.lora_A.to(torch.bfloat16); m.lora_B.to(torch.bfloat16)
    if same_weights is not None:  # the b200 arm's adapters (fp32 masters -> the bf16 values its kernels read)
        for m, (A, Bm) in zip(wrapped, same_weights["adapters"]):
            with torch.no_grad():
                m.lora_A["default"].weight.copy_(A.to(torch.bfloat16))
                m.lora_B["default"].weight.copy_(Bm.to(torch.bfloat16))
    unet.train()
    sched = make_scheduler(kind, dev) if kind != "dreambooth" else None
    d = {k: v.to(dev) for k, v in host.items()}
    accum = 4 if kind == "dreambooth" else ACCUM

    def one():
        for m in wrapped:
            m.lora_A["default"].weight.grad = None
            m.lora_B["default"].weight.grad = None
        if kind == "dreambooth":
            return micro_step.oracle_dreambooth_micro_step(olora, olosses, unet, d, loss_type="pso", beta_pso=5.0, neg_defactor=0.1,
                                                           prior_loss_weight=0.5, loss_scale=1.0 / accum)[0].detach()
        return micro_step.oracle_micro_step(olora, olosses, unet, d, sched, beta=50.0, eps=0.1, loss_scale=1.0 / ACCUM,
                                            kind=kind).detach()  # no autograd graph kept alive between steps

    def timed(fn, n):
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(n + 1)]
        torch.cuda.synchronize()
        evs[0].record()
        for i in range(n):
            fn()
            evs[i + 1].record()
        torch.cuda.synchronize()
        return statistics.mean(evs[i].elapsed_time(evs[i + 1]) for i in range(n))
    B = args.pairs
    side = torch.cuda.Stream()  # everything on ONE non-default stream: the AccumulateGrad nodes are created under it
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            loss = one()
        ms_eager = timed(one, reps)
        out = {"kind": "torch-eager on this GPU: stock nn.Linear + peft-style LoRA module (3 cuBLAS GEMMs + scale + add), 4 "
                       "forwards, ~340-launch loss chain, autograd; bf16, activations resident",
               "value": round(B / (ms_eager * 1e-3), 3), "unit": UNIT, "ms_per_step": round(ms_eager, 2), "steps": reps,
               "loss": round(float(loss.item()) * accum, 6)}
        if kind != "turbo":  # the same step replayed from a CUDA graph (no host launch latency); the Turbo flow syncs (.item(), TS:63)
            try:
                graph = torch.cuda.CUDAGraph()
                torch.cuda.synchronize()
                with torch.cuda.graph(graph, stream=side):
                    one()
                graph.replay()
                ms_graph = timed(graph.replay, reps)
                out["graph_replayed"] = {"value": round(B / (ms_graph * 1e-3), 3), "ms_per_step": round(ms_graph, 2)}
                del graph
            except Exception as e:
                out["graph_replayed"] = {"unavailable": f"{type(e).__name__}: {str(e)[:160]}"}
        else:
            out["graph_replayed"] = {"unavailable": "the Euler-ancestral step of the reference syncs with the host once per sample "
                                                    "(turbo_inference_with_logprob.py:63): not capturable"}
    torch.cuda.synchronize()
    if same_weights is not None:
        # same weights, same batch, one micro-step: the reference's flow on stock kernels vs this repo's kernels
        with torch.cuda.stream(side):
            loss_e = float(one().item()) * accum
        torch.cuda.synchronize()
        g_ours = same_weights["grad"].double()
        g_eager = torch.zeros_like(g_ours)
        for m, (oa, ob) in zip(wrapped, same_weights["order"]):
            ga, gb = m.lora_A["default"].weight.grad, m.lora_B["default"].weight.grad
            g_eager[oa:oa + ga.numel()] = ga.double().flatten()
            g_eager[ob:ob + gb.numel()] = gb.double().flatten()
        cos = float((torch.dot(g_ours, g_eager) / (g_ours.norm() * g_eager.norm())).item())
        out["same_weights_parity"] = {
            "what": "one micro-step of both arms on the SAME base weights, adapters and batch (bf16 both; the eager arm also keeps "
                    "its adapter gradients in bf16): the reference's flow on stock torch kernels vs this repo's kernels",
            "loss_ours": round(same_weights["loss"], 6), "loss_eager": round(loss_e, 6),
            "loss_rel_diff": round(abs(same_weights["loss"] - loss_e) / abs(loss_e), 6),
            "grad_cosine": round(cos, 6), "grad_norm_ratio": round(float((g_ours.norm() / g_eager.norm()).item()), 5)}
        del g_ours, g_eager
    del unet, wrapped
    import gc
    gc.collect()
    torch.cuda.empty_cache()
    return out


def run_b200(args):
    import pairwise_sample_optimization_b200 as pso
    from pairwise_sample_optimization_b200 import _lib

    rank, world, local = dist_env()
    if args.gpus != world and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback for the b200 arm")
    L = _lib.lib()  # fail loudly if the CUDA library is missing
    if args.deterministic:  # what torch's deterministic mode needs before the first cuBLAS call (B200Arm switches the mode)
        os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")  # 8 x 4 MiB: a fixed cuBLAS workspace per stream
        torch.utils.deterministic.fill_uninitialized_memory = False  # no NaN fill of every torch.empty: not needed for that
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    K, W = args.steps, max(args.warmup, 3)
    peaks = measured_peaks()

    arm = B200Arm(args, args.config, dev, rank, world, L)
    if not args.no_graph:
        arm.capture()
    t = arm.timed(K, W)
    if args.dump_outputs and rank == 0:
        arm.dump_outputs(args.dump_outputs)
    e2e = arm.e2e(K)
    peak_hbm_gb = round(torch.cuda.max_memory_allocated(dev) / 2 ** 30, 2)  # before the second (instrumented) graph
    roofline, skinny = arm.instrumented(t["ms_per_step"], peaks)
    gate = arm.gate()
    extra = {}
    if world > 1:
        extra["exchange_check"] = arm.exchange_check()
    run_details = {"parallelism": f"dp{world} (pairs sharded; one exchange of the flat LoRA gradient per {arm.accum} steps)",
                   "gradient_exchange": arm.exchange_kind,
                   "activations": ("recomputed in the backward (gradient checkpointing, as the reference)" if args.grad_checkpointing
                                   else "resident in HBM (no gradient checkpointing: same gradients, no recompute forward)"),
                   "weight_gradients": "dA / dB launches on a side stream" if args.wgrad_stream else "in stream order",
                   "projections": ("q / k / v (k / v) stacked: one launch per group and direction, t / u as tiles of the main "
                                   "launch" if args.fuse_projections else "one launch sequence per projection"),
                   "cross_attention_kv": ("k / v of all cross-attention layers in one launch per shape at forward start (they read "
                                          "the prompt embeddings only); backward per layer" if (args.kv_bank and args.fuse_projections)
                                          else "per block"),
                   "feed_forward": "fused GEGLU kernels" if args.fused_geglu else "stock torch GEGLU",
                   "l2_policy": "working set larger than L2 (5.1 GB of bf16 weights streamed every forward)",
                   "forwards": "4 separate (as the reference)" if args.separate_forwards else
                               "win+lose batched: 1 policy + 1 reference forward of batch 2B" +
                               (", reference forward on a second stream" if arm.ref_stream is not None else ""),
                   "timing": ("eager launches" if args.no_graph else "micro-step replayed from one CUDA graph; optimizer "
                              "boundary eager") + ", CUDA events around K steps, max over ranks"}
    host_batch = {k: v.clone() for k, v in arm.host.items()}
    # the adapters and one micro-step's loss / flat gradient of this arm: the eager baseline re-runs the reference's flow on the
    # SAME weights and batch and reports how far the two arms are apart (end-to-end parity at the full SDXL-architecture size)
    same_weights = None
    if rank == 0 and world == 1 and not args.no_eager_baseline and arm.one_step is not None:
        same_weights = {"adapters": [(m.lora_A["default"].weight.detach().clone(), m.lora_B["default"].weight.detach().clone())
                                     for m in lora_layers_in_module_order(arm.unet)],
                        "loss": arm.one_step["loss"], "grad": arm.one_step["grad"], "order": flat_order(arm)}
    arm.close()
    del arm

    def guarded(key, fn):
        """Optional blocks never cost the headline line: a failure is recorded under the block's key."""
        try:
            extra[key] = fn()
        except Exception as e:  # noqa: BLE001
            import traceback
            traceback.print_exc()
            extra[key] = {"error": f"{type(e).__name__}: {str(e)[:200]}"}
            torch.cuda.synchronize()

    if rank == 0 and not args.no_kernel_figures:
        guarded("loss_kernel_roofline", lambda: loss_kernel_roofline(pso, dev, peaks))
        guarded("sampler_kernel_roofline", lambda: sampler_kernel_roofline(dev, peaks))
        guarded("lora_gemm_large", lambda: lora_gemm_large(dev, peaks))
        if args.config == "dmd128" and not args.tiny:
            guarded("lora_projection_vs_cublas", lambda: lora_projection_vs_cublas(
                dev, [(8192, 1280, 1280), (32768, 640, 640), (616, 2048, 1280)], CONFIGS[args.config]["rank"]))
    if world == 1 and args.config == "dmd128" and not args.no_turbo64 and not args.tiny:
        # configs[1], short: the latency-bound regime (M = 2048 launches), driver-visible next to the headline configuration
        def turbo64_block():
            arm2 = B200Arm(args, "turbo64", dev, rank, world, L)
            try:
                if not args.no_graph:
                    arm2.capture()
                t2 = arm2.timed(6, 3)
                r2, s2 = arm2.instrumented(t2["ms_per_step"], peaks)
                for blk in (r2, s2):
                    blk.pop("how", None); blk.pop("by_launch", None)
                return {"config": config_block(args, "turbo64"), "value": round(t2["value"], 3), "unit": UNIT, "steps": 6,
                        "warmup": 3, "ms_per_step": round(t2["ms_per_step"], 3), "gpu_launches": t2["launches"],
                        "loss": round(t2["loss"], 6), "roofline": r2, "lora_skinny_launches": s2}
            finally:
                arm2.close()
        guarded("turbo64", turbo64_block)
    if rank == 0 and world == 1 and not args.no_eager_baseline:
        def eager_block():
            eager = gpu_eager_baseline(args, args.config, dev, host_batch, same_weights=same_weights)
            eager["ratio_ours_over_eager"] = round(t["value"] / eager["value"], 3)
            if "value" in eager.get("graph_replayed", {}):
                eager["ratio_ours_over_graph_replayed"] = round(t["value"] / eager["graph_replayed"]["value"], 3)
            return eager
        guarded("gpu_eager_baseline", eager_block)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_reference(args, reps=1, warmup=0)
    if rank == 0:
        line = {
            "metric": METRIC, "value": round(t["value"], 3), "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": round(t["ms_per_step"], 3), "ms_per_step_each": [round(v, 1) for v in t["per_step"]],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic",
            "config": config_block(args, args.config), "run_details": run_details,
            "gpu_launches": t["launches"], "clocks": t["clocks"], "e2e": e2e, "roofline": roofline,
            "lora_skinny_launches": skinny,
            "loss": round(t["loss"], 6), "grad_norm": t.get("grad_norm"), "gate": gate, "peak_hbm_gb": peak_hbm_gb,
        }
        line.update(extra)
        if cpu is not None:
            line["cpu_baseline"] = cpu
        print(json.dumps(line), flush=True)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


# ----------------------------------------------------------------------------------------------- reference arm (CPU)
def _make_cpu_step(args, pairs):
    """The reference's micro-step restated with the oracle pieces (oracle/ is checker code; it is executed here only as
    the reported CPU baseline / reference arm): fp32, same UNet architecture, oracle LoRA modules (peft forward restated),
    four step-with-logprob calls, the inline loss, autograd backward; all host threads."""
    from fixtures import micro_step, sdxl_unet
    from oracle import lora as olora, losses as olosses, schedules
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    cfg = sdxl_unet.tiny_config() if args.tiny else sdxl_unet.sdxl_config()
    with torch.device("meta"):
        unet = sdxl_unet.UNet2DConditionModel(cfg)
    unet = unet.to_empty(device="cpu")
    g = torch.Generator().manual_seed(0)
    pool = torch.randn(1 << 22, generator=g) * 0.02  # cheap random init: values only need to be finite and small
    with torch.no_grad():
        for prm in unet.parameters():
            n = prm.numel()
            flat = prm.view(-1)
            for off in range(0, n, pool.numel()):
                m = min(pool.numel(), n - off)
                flat[off:off + m] = pool[:m]
            if prm.dim() == 1:
                prm.zero_()
        for mod in unet.modules():
            if isinstance(mod, (torch.nn.GroupNorm, torch.nn.LayerNorm)):
                mod.weight.fill_(1.0)
                mod.bias.zero_()
    unet.requires_grad_(False)
    conf = CONFIGS[args.config]
    KIND, LATENT_HW, RANK = conf["kind"], conf["latent_hw"], conf["rank"]
    wrapped = olora.oracle_add_adapter(unet, RANK, RANK)
    for m in wrapped:
        torch.nn.init.normal_(m.lora_B["default"].weight, std=0.01)
    unet.train()
    unet.enable_gradient_checkpointing()
    pooled = cfg.projection_class_embeddings_input_dim - 6 * cfg.addition_time_embed_dim
    if KIND == "dreambooth":
        sched = schedules.dreambooth_scheduler()
        batch = micro_step.synth_dreambooth_batch(pairs, LATENT_HW, cfg.cross_attention_dim, pooled, 100, sched)
    else:
        sched = schedules.turbo_scheduler(4) if KIND == "turbo" else schedules.dmd_scheduler()
        batch = micro_step.synth_batch(pairs, LATENT_HW, cfg.cross_attention_dim, pooled, 100, getattr(sched, "sigmas", None),
                                       kind=KIND)

    def one():
        if KIND == "dreambooth":
            loss, _ = micro_step.oracle_dreambooth_micro_step(olora, olosses, unet, batch, loss_type="pso", beta_pso=5.0,
                                                              neg_defactor=0.1, prior_loss_weight=0.5, loss_scale=0.25)
            scale = 4
        else:
            loss = micro_step.oracle_micro_step(olora, olosses, unet, batch, sched, beta=50.0, eps=0.1, loss_scale=1.0 / ACCUM,
                                                kind=KIND)
            scale = ACCUM
        for m in wrapped:
            m.lora_A["default"].weight.grad = None
            m.lora_B["default"].weight.grad = None
        return float(loss.detach()) * scale
    return one, threads


def cpu_reference(args, reps, warmup):
    pairs = args.cpu_pairs
    one, threads = _make_cpu_step(args, pairs)
    for _ in range(warmup):
        one()
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        one()
        times.append(time.perf_counter() - t0)
    med = statistics.median(times)
    return {"value": round(pairs / med, 4), "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{pairs} pair(s) x {len(times)} rep(s) of the same micro-step (fp32, torch {torch.__version__} CPU, "
                      f"{torch.get_num_threads()} threads, no warm-up), {med:.1f} s per step",
            "ms_per_step": round(med * 1e3, 1)}


def run_reference(args):
    rank, world, _ = dist_env()
    if rank != 0:
        return
    K, W = args.steps, min(args.warmup, 1)
    pairs = args.cpu_pairs
    one, threads = _make_cpu_step(args, pairs)
    t_begin = time.perf_counter()
    res = None
    for _ in range(W):
        res = one()
    times = []
    for _ in range(K):  # each step: one micro-step over `pairs` pair(s); bounded by --ref-budget-seconds
        t0 = time.perf_counter()
        res = one()
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_begin > args.ref_budget_seconds:
            break
    ms = statistics.mean(times) * 1e3
    value = pairs / (ms * 1e-3)
    sample = (f"{pairs} pair(s) per step (bounded sample of the {args.pairs}-pair micro-step), fp32, torch {torch.__version__} CPU, "
              f"{torch.get_num_threads()} threads; {len(times)} of the {K} requested steps fit the {args.ref_budget_seconds:.0f} s budget")
    line = {"impl": "reference", "metric": METRIC, "value": round(value, 4), "unit": UNIT, "n_gpus": args.gpus,
            "steps": len(times), "steps_requested": K, "warmup": W, "ms_per_step": round(ms, 1), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_block(args, args.config),
            "run_details": {"arm": "oracle port of the reference's PyTorch path on the host cores (fp32, gradient checkpointing "
                                   "on as the reference ships it)", "pairs_per_step_sample": pairs},
            "cpu_baseline": {"value": round(value, 4), "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": round(value, 4), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "loss": round(res, 6)}
    print(json.dumps(line), flush=True)


def parse_args(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=12)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="dmd128", choices=sorted(CONFIGS),
                    help="dmd128 = the configuration BASELINE.json's metric is quoted on (SDXL 128x128 latents); turbo64 = configs[1]")
    ap.add_argument("--pairs", type=int, default=4, help="pairs per GPU per micro-step (train.batch_size of the shipped recipe)")
    ap.add_argument("--cpu-pairs", type=int, default=1, help="pairs in the bounded CPU sample")
    ap.add_argument("--ref-budget-seconds", type=float, default=150.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-kernel-figures", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch the micro-step eagerly instead of replaying a CUDA graph")
    ap.add_argument("--separate-forwards", action="store_true", help="4 UNet forwards of batch B instead of 2 of batch 2B")
    ap.add_argument("--overlap-reference", action="store_true", default=True,
                    help="issue the frozen-reference forward on a second stream (default)")
    ap.add_argument("--no-overlap-reference", dest="overlap_reference", action="store_false")
    ap.add_argument("--grad-checkpointing", dest="grad_checkpointing", action="store_true", default=False,
                    help="recompute the blocks in the backward (the reference's memory workaround, turbo trainer :358); default: "
                         "the activations of the 4-pair micro-step (43 GB at 128x128 latents) stay resident in the 180 GB of HBM")
    ap.add_argument("--no-grad-checkpointing", dest="grad_checkpointing", action="store_false")
    ap.add_argument("--wgrad-stream", dest="wgrad_stream", action="store_true", default=True,
                    help="issue the dA / dB launches of every projection on a side stream (joined at the end of the backward)")
    ap.add_argument("--no-wgrad-stream", dest="wgrad_stream", action="store_false")
    ap.add_argument("--exchange", default="multimem", choices=["multimem", "nccl"],
                    help="N > 1: the LoRA-gradient exchange (multimem = this repo's NVLink-multicast kernel; nccl = ncclAllReduce)")
    ap.add_argument("--no-fused-geglu", dest="fused_geglu", action="store_false", default=True,
                    help="leave the feed-forward's GEGLU on the stock torch kernels")
    ap.add_argument("--tiny", action="store_true", help="debug: the 32/64-channel fixture instead of the SDXL architecture")
    ap.add_argument("--no-fuse-projections", dest="fuse_projections", action="store_false", default=True,
                    help="one launch sequence per projection instead of stacked q / k / v (k / v) groups")
    ap.add_argument("--no-kv-bank", dest="kv_bank", action="store_false", default=True,
                    help="A/B: cross-attention k / v projections launched per block instead of once per forward for all blocks")
    ap.add_argument("--programmatic-launch", action="store_true",
                    help="A/B: projection kernels launched with programmatic stream serialization (prologue overlaps the "
                         "preceding kernel's tail)")
    ap.add_argument("--no-inlaunch-deps", action="store_true",
                    help="A/B: t / u as launches of their own (PDL overlap) instead of tiles of the main launch")
    ap.add_argument("--profiler-range", action="store_true",
                    help="cudaProfilerStart/Stop around the last timed step (for `ncu --profile-from-start off` launch lists; "
                         "the printed numbers of such a run are not bench values)")
    ap.add_argument("--no-eager-baseline", action="store_true", help="skip the torch-eager-on-this-GPU baseline")
    ap.add_argument("--no-turbo64", action="store_true", help="skip the short configs[1] block after the main timing")
    ap.add_argument("--deterministic", action=argparse.BooleanOptionalAction, default=True,
                    help="this library's arms (headline, turbo64) with unsplit dA / dB reductions and torch's deterministic "
                         "algorithms: the same arguments give the same outputs (default); --no-deterministic times the library "
                         "defaults, whose outputs vary from run to run in the last bits (amplified by AdamW). The stock-torch "
                         "arms always run torch's defaults")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the loss, gradient norm and (sampled) flat LoRA buffers the last timed step left, as DIR/<name>.npy")
    return ap.parse_args(argv)


def main():
    args = parse_args()
    if args.impl == "reference":
        if args.dump_outputs:
            raise SystemExit("--dump-outputs writes the b200 arm's outputs; run it without --impl reference")
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()

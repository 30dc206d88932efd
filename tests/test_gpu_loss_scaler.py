"""Device-resident dynamic loss scaling (``amp.DeviceGradScaler``, torch's GradScaler semantics) through the fused losses
and the optimizer boundary: the scaled loss gradient is S x the unscaled one (and rounded once, already scaled, in fp16),
the scale update equals torch._amp_update_scale_, the boundary tracks GradScaler + clip_grad_norm_ + AdamW and the 8-bit
oracle, a scaler at S = 1 changes nothing, CUDA-graph replays follow the device scale, checkpoints carry it, the fp16 tiny
UNet runs through overflow back-off, and two ranks agree."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import loss_scaler as ols, make_golden, optim8bit as o8
from tests import _util as U

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HYPER = dict(lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2, max_grad_norm=1.0)


@pytest.fixture(scope="module")
def pso(built_lib):
    import pairwise_sample_optimization_b200 as m
    return m


def _scaler(pso, init_scale, **kw):
    return pso.DeviceGradScaler("cuda", init_scale=init_scale, **kw)


def _online(pso, d, scaler=None, tune=(0, 0), scaled_backward=True):
    pred = [U.cuda(p).requires_grad_(True) for p in d["noise_pred"]]
    loss, st = pso.pso_pair_loss(pred[0], pred[1], U.cuda(d["noise_ref_pred"][0]), U.cuda(d["noise_ref_pred"][1]),
                                 U.cuda(d["latents"][0]), U.cuda(d["latents"][1]), U.cuda(d["next_latents"][0]),
                                 U.cuda(d["next_latents"][1]), U.cuda(d["timesteps"][0]), U.cuda(d["timesteps"][1]),
                                 U.cuda(d["human_prefer"]), scheduler=d["sched"], kind=d["kind"], step_ratio=d["step_ratio"],
                                 return_stats=True, tune=tune, grad_scaler=scaler)
    (scaler.scale(loss) if scaler is not None and scaled_backward else loss).backward()
    return loss.detach(), st, pred[0].grad, pred[1].grad


def _same_bits(a, b):
    return torch.equal(a.view(torch.int32) if a.dtype == torch.float32 else a, b.view(torch.int32) if b.dtype == torch.float32 else b)


# ----------------------------------------------------------------------------------------------- loss side
@pytest.mark.parametrize("S", [2.0 ** 10, 2.0 ** 16])
@pytest.mark.parametrize("kind", ["turbo", "dmd"])
@pytest.mark.parametrize("shape,tune", [((4, 64, 64), (0, 0)), ((4, 9, 9), (0, 0)), ((4, 64, 64), (256, 0))],
                         ids=["tmem", "ragged", "general"])
def test_online_scaled_gradient_is_S_times_the_unscaled_one(pso, S, kind, shape, tune):
    d = U.synth(kind, 3, shape, 7)
    l0, s0, a0, b0 = _online(pso, d, tune=tune)
    sc = _scaler(pso, S)
    l1, s1, a1, b1 = _online(pso, d, sc, tune=tune)
    assert float(a0.abs().max()) > 0 and float(b0.abs().max()) > 0
    assert _same_bits(l0, l1) and _same_bits(s0, s1)  # loss and stats stay unscaled
    assert _same_bits(a1, a0 * S) and _same_bits(b1, b0 * S)
    assert sc.get_scale() == S  # the loss never changes the scale
    # a plain loss.backward() with a scaler gives the unscaled gradient back (upstream factor 1 / S on the device)
    l2, _, a2, b2 = _online(pso, d, sc, tune=tune, scaled_backward=False)
    assert _same_bits(l2, l0) and _same_bits(a2, a0) and _same_bits(b2, b0)


@pytest.mark.parametrize("loss_type", ["pso", "pso_db"])
@pytest.mark.parametrize("shape", [(4, 64, 64), (4, 9, 9)], ids=["tmem", "ragged"])
def test_dreambooth_scaled_gradient_is_S_times_the_unscaled_one(pso, loss_type, shape):
    db = make_golden.synth_dreambooth(2, shape, 4)
    S = 2.0 ** 16

    def run(scaler):
        mp = db["model_pred"].cuda().requires_grad_(True)
        out = pso.pso_db_loss(mp, db["ref_pred"].cuda() if loss_type == "pso" else None, db["noisy"].cuda(), db["x0"].cuda(),
                              db["sigmas"].cuda(), loss_type=loss_type, beta_pso=5.0, neg_defactor=0.1, prior_loss_weight=0.5,
                              grad_scaler=scaler)
        (scaler.scale(out[0]) if scaler is not None else out[0]).backward()
        return [t.detach() for t in out], mp.grad

    (l0, *st0), g0 = run(None)
    (l1, *st1), g1 = run(_scaler(pso, S))
    assert float(g0.abs().max()) > 0
    assert _same_bits(l0, l1) and all(_same_bits(a, b) for a, b in zip(st0, st1))
    assert _same_bits(g1, g0 * S)


@pytest.mark.parametrize("kind", ["turbo", "dmd"])
def test_fp16_gradient_is_rounded_once_after_scaling(pso, kind, monkeypatch):
    """fp16 predictions, a few percent of the per-element gradients below fp16's normal range (6.1e-5): the kernel's
    gradient is within 1 ulp of S x the fp64 closed form; scaler.scale(loss).backward() hands exactly that to autograd;
    loss.backward() the unscaled one."""
    from pairwise_sample_optimization_b200 import losses
    d = U.synth(kind, 2, (4, 64, 64), 3, pred_dtype=torch.float16, latent_dtype=torch.float16)
    cf = U.oracle_fp64(d)
    S = 2.0 ** 16
    assert max(g.abs().max().item() for g in cf["grads"]) * S < 6.0e4  # scaled: finite in fp16
    assert all(float(((g != 0) & (g.abs() < 6.1e-5)).double().mean()) > 0.01 for g in cf["grads"])  # unscaled: subnormal
    seen = []
    orig = losses._apply_upstream

    def spy(grads, grad_out, dev, scaler=None):
        seen.append([g.clone() for g in grads])  # what the kernel wrote, before the upstream factor
        return orig(grads, grad_out, dev, scaler)

    monkeypatch.setattr(losses, "_apply_upstream", spy)
    _, _, a1, b1 = _online(pso, d, _scaler(pso, S))
    for k, got in enumerate((a1, b1)):
        assert torch.equal(got, seen[0][k])  # the upstream factor S / S = 1 changed nothing
        U.assert_rounded_equal(got, cf["grads"][k] * S, torch.float16)
    _, _, a2, b2 = _online(pso, d, _scaler(pso, S), scaled_backward=False)
    for k, got in enumerate((a2, b2)):
        U.assert_rounded_equal(got, cf["grads"][k], torch.float16)


# ----------------------------------------------------------------------------------------------- optimizer boundary
def _lora_model(L, r=4, seed=3):
    from tests.test_gpu_lora import _Attention
    torch.manual_seed(seed)
    m = _Attention(640, 2048, 10, 64).to(device="cuda", dtype=torch.bfloat16)
    for w in L.add_adapter(m, L.LoraConfig(r=r, lora_alpha=r)):
        torch.nn.init.normal_(w.lora_B["default"].weight, std=0.05)
    return m


def _opt(pso, bits, scaler=None, seed=3, **kw):
    L = pso.lora
    m = _lora_model(L, seed=seed)
    extra = dict(optim_bits=8, min_8bit_size=1024) if bits == 8 else {}
    return m, L.FusedLoRAOptimizer(m, **HYPER, **extra, grad_scaler=scaler, **kw)


def _moments(opt):
    if opt.optim_bits == 32:
        return [opt.exp_avg, opt.exp_avg_sq]
    return [opt.code1, opt.code2, opt.absmax1, opt.absmax2, opt.exp_avg32, opt.exp_avg_sq32]


def _snapshot(opt):
    return [t.clone() for t in [opt.flat_param, opt.flat_operand, *_moments(opt)]]


INJECT = {2: float("inf"), 7: float("inf"), 8: float("nan")}


@pytest.mark.parametrize("bits", [32, 8])
@pytest.mark.parametrize("growth,backoff", [(2.0, 0.5), (1.3, 0.7)])
def test_scale_update_matches_torch_amp_update_scale(pso, bits, growth, backoff):
    sc = _scaler(pso, 2.0 ** 12, growth_factor=growth, backoff_factor=backoff, growth_interval=3)
    _, opt = _opt(pso, bits, sc)
    want_s = torch.full((1,), 2.0 ** 12, device="cuda")
    want_t = torch.zeros(1, dtype=torch.int32, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(1)
    n = opt.flat_param.numel()
    for b in range(12):
        opt.bucket.flat.copy_(torch.randn(n, device="cuda", generator=g) * 1e-3 * sc.scale_tensor)
        if b in INJECT:
            opt.bucket.flat[n // 3] = INJECT[b]
        before = _snapshot(opt)
        opt.step()
        torch._amp_update_scale_(want_s, want_t, opt.found_inf, growth, backoff, 3)
        assert float(opt.found_inf) == (1.0 if b in INJECT else 0.0), b
        assert _same_bits(sc.scale_tensor, want_s) and torch.equal(sc.growth_tracker, want_t), b
        if b in INJECT:
            assert all(torch.equal(x, y) for x, y in zip(before, _snapshot(opt))), f"boundary {b} moved the state"
        assert float(opt.bucket.flat.abs().max()) == 0.0
    assert int(opt.step_dev.item()) == 12 - len(INJECT)
    assert sc.get_scale() != 2.0 ** 12  # it grew and backed off on the way


def test_boundary_tracks_torch_gradscaler_clip_and_adamw(pso):
    """GradScaler("cuda") + unscale_ + clip_grad_norm_ + AdamW per parameter on the same scaled gradients: identical skip
    pattern and scale, parameters within the fp32 parity tolerance of the unscaled boundary."""
    L = pso.lora
    sc = _scaler(pso, 2.0 ** 10, growth_interval=2)
    attn, opt = _opt(pso, 32, sc)
    params = L.lora_parameters(attn)
    ref = [p.detach().clone().requires_grad_(True) for p in params]
    ref_opt = torch.optim.AdamW(ref, lr=HYPER["lr"], betas=HYPER["betas"], eps=HYPER["eps"], weight_decay=HYPER["weight_decay"])
    ts = torch.amp.GradScaler("cuda", init_scale=2.0 ** 10, growth_interval=2)
    g = torch.Generator(device="cuda").manual_seed(5)
    for b in range(8):
        S = sc.get_scale()
        assert S == ts.get_scale(), b
        for i, (p, q) in enumerate(zip(params, ref)):
            grad = torch.randn(p.shape, device="cuda", generator=g) * (3.0 if b == 0 else 0.01) * S
            if b == 3 and i == 1:
                grad[0, 0] = float("inf")
            if b == 5 and i == 4:
                grad[0, 0] = float("nan")
            p.grad.copy_(grad)
            q.grad = grad.clone()
        ts.scale(torch.zeros((), device="cuda"))  # a training loop's scaler.scale(loss) (torch initialises its state there)
        ts.unscale_(ref_opt)
        torch.nn.utils.clip_grad_norm_(ref, HYPER["max_grad_norm"])
        ts.step(ref_opt)
        ts.update()
        opt.step()
        assert float(opt.found_inf) == (1.0 if b in (3, 5) else 0.0), b
        assert sc.get_scale() == ts.get_scale(), b
        for p, q in zip(params, ref):
            assert (p.detach() - q.detach()).abs().max().item() <= 2e-6 * max(q.detach().abs().max().item(), 1e-3), b


def test_8bit_boundary_is_bitwise_the_oracle_with_the_unscale_factor(pso):
    sc = _scaler(pso, 2.0 ** 14, growth_interval=2)
    _, opt = _opt(pso, 8, sc)
    blocks8, chunks32 = opt.blocks8.cpu().numpy(), opt.chunks32.cpu().numpy()
    st = {k: getattr(opt, k).cpu().numpy().copy() for k in ("code1", "code2", "absmax1", "absmax2", "exp_avg32",
                                                            "exp_avg_sq32", "qmap1", "qmap2")}
    p = opt.flat_param.cpu().numpy().copy()
    gen = torch.Generator().manual_seed(9)
    t = 0
    for b in range(5):
        S = np.float32(sc.get_scale())
        grad = (torch.randn(p.shape[0], generator=gen) * (3.0 if b == 0 else 1e-3) * float(S)).numpy()
        if b == 2:
            grad[77] = np.inf
        opt.bucket.flat.copy_(torch.from_numpy(grad))
        norm = opt.step().item()
        t += 0 if b == 2 else 1
        p, st = o8.adamw8_step(st, p, grad, blocks8, chunks32, norm, t, HYPER["lr"], *HYPER["betas"], HYPER["eps"],
                               HYPER["weight_decay"], HYPER["max_grad_norm"], grad_scale=float(ols.unscale_factor(S)))
        assert np.array_equal(opt.flat_param.cpu().numpy(), p), b
        for k in st:
            assert np.array_equal(getattr(opt, k).cpu().numpy(), st[k]), (b, k)
    assert sc.get_scale() != 2.0 ** 14


@pytest.mark.parametrize("bits", [32, 8])
def test_a_scaler_that_stays_at_one_changes_nothing(pso, bits):
    sc = _scaler(pso, 1.0, growth_interval=2 ** 30)
    _, a = _opt(pso, bits, sc)
    _, b = _opt(pso, bits)
    gen = torch.Generator(device="cuda").manual_seed(4)
    for k in range(4):
        grad = torch.randn(a.flat_param.numel(), device="cuda", generator=gen) * (3.0 if k == 0 else 1e-3)
        for o in (a, b):
            o.bucket.flat.copy_(grad)
        na, nb = a.step().clone(), b.step().clone()
        assert _same_bits(na, nb)
        assert all(torch.equal(x, y) for x, y in zip(_snapshot(a), _snapshot(b))), k
    assert sc.get_scale() == 1.0 and int(sc.growth_tracker.item()) == 4


def test_cuda_graph_replays_follow_the_device_scale(pso):
    """One captured micro-step (LoRA projection -> fused loss, scaler.scale(loss).backward()) + step(), replayed with an
    overflow injected on one replay: gradients, S, tracker and parameters equal the eager run step for step."""
    L = pso.lora
    L.set_deterministic_wgrad(True)
    try:
        B, M = 2, 64
        g = torch.Generator(device="cuda").manual_seed(0)
        xs = [torch.randn(B, M, 640, device="cuda", generator=g).bfloat16() for _ in range(2)]
        refs = [torch.randn(B, M, 640, device="cuda", generator=g).bfloat16() * 0.1 for _ in range(2)]
        lat = [torch.randn(B, M, 640, device="cuda", generator=g).bfloat16() for _ in range(4)]
        coef = [tuple(torch.full((B,), v, device="cuda") for v in (1.0, -0.5, 0.3)) for _ in range(2)]
        hp = torch.tensor([[-1.0, 1.0], [1.0, -1.0]], device="cuda")

        def make():
            sc = _scaler(pso, 2.0 ** 8, growth_interval=2)
            m = _lora_model(L, seed=11)
            return m, sc, L.FusedLoRAOptimizer(m, **HYPER, grad_scaler=sc)

        def micro(m, sc, opt, snap):
            p0, p1 = m.to_q(xs[0]), m.to_q(xs[1])
            loss = pso.pso_pair_loss(p0, p1, refs[0], refs[1], lat[0], lat[1], lat[2], lat[3], None, None, hp, kind="affine",
                                     coefficients=coef, beta=5.0, grad_scaler=sc)
            sc.scale(loss).backward()
            snap.copy_(opt.bucket.flat)
            opt.step()

        eager, graphed = make(), make()
        snaps = [torch.zeros_like(eager[2].bucket.flat), torch.zeros_like(graphed[2].bucket.flat)]
        for (m, sc, opt), s in zip((eager, graphed), snaps):  # warm-up: lazy kernel configuration happens outside capture
            micro(m, sc, opt, s)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            micro(*graphed, snaps[1])
        seen = [graphed[1].get_scale()]
        for k in range(6):
            for o in (eager[2], graphed[2]):
                if k == 3:
                    o.bucket.flat[5] = float("inf")
            micro(*eager, snaps[0])
            graph.replay()
            torch.cuda.synchronize()
            assert _same_bits(snaps[0], snaps[1]), k
            assert _same_bits(eager[1].scale_tensor, graphed[1].scale_tensor), k
            assert torch.equal(eager[1].growth_tracker, graphed[1].growth_tracker), k
            assert torch.equal(eager[2].flat_param, graphed[2].flat_param), k
            assert float(graphed[2].found_inf) == (1.0 if k == 3 else 0.0)
            seen.append(graphed[1].get_scale())
        # the replays read a scale that kept changing: growth every second finite replay, back-off on the overflow
        assert sum(a != b for a, b in zip(seen, seen[1:])) >= 3, seen
    finally:
        L.set_deterministic_wgrad(False)


def test_checkpoint_carries_the_scaler_and_refuses_to_drop_it(pso, tmp_path):
    from safetensors import safe_open

    from pairwise_sample_optimization_b200 import _lib, checkpoint
    sc = _scaler(pso, 2.0 ** 12, growth_factor=1.5, growth_interval=3)
    attn, opt = _opt(pso, 32, sc)
    gen = torch.Generator(device="cuda").manual_seed(6)
    grads = [torch.randn(opt.flat_param.numel(), device="cuda", generator=gen) * 1e-3 for _ in range(6)]
    for k in range(4):
        opt.bucket.flat.copy_(grads[k] * sc.scale_tensor)
        if k == 1:
            opt.bucket.flat[3] = float("inf")
        opt.step()
    checkpoint.save_state(str(tmp_path), attn, opt)
    with safe_open(os.path.join(str(tmp_path), checkpoint.OPTIMIZER_NAME), framework="pt") as f:
        keys, meta = set(f.keys()), f.metadata()
    assert keys == {"flat_param", "exp_avg", "exp_avg_sq", "scaler_scale", "scaler_growth_tracker"}
    assert "scaler" in meta
    sc2 = _scaler(pso, 1.0)
    attn2, opt2 = _opt(pso, 32, sc2, seed=99)
    checkpoint.load_state(str(tmp_path), attn2, opt2)
    assert sc2.state_dict() == sc.state_dict()
    for k in (4, 5):
        for o, s in ((opt, sc), (opt2, sc2)):
            o.bucket.flat.copy_(grads[k] * s.scale_tensor)
            o.step()
        assert torch.equal(opt.flat_param, opt2.flat_param) and torch.equal(opt.exp_avg_sq, opt2.exp_avg_sq)
        assert _same_bits(sc.scale_tensor, sc2.scale_tensor) and torch.equal(sc.growth_tracker, sc2.growth_tracker)
    # scaler state but no scaler attached: refused, not dropped
    _, plain = _opt(pso, 32)
    with pytest.raises(_lib.Psob200Error, match="grad_scaler"):
        checkpoint.load_optimizer_state(str(tmp_path), plain)
    # no scaler in the file: an attached scaler keeps its values; the file without a scaler has today's keys
    checkpoint.save_optimizer_state(str(tmp_path / "plain"), plain)
    with safe_open(os.path.join(str(tmp_path / "plain"), checkpoint.OPTIMIZER_NAME), framework="pt") as f:
        assert set(f.keys()) == {"flat_param", "exp_avg", "exp_avg_sq"} and "scaler" not in f.metadata()
    sc3 = _scaler(pso, 512.0, growth_interval=7)
    _, opt3 = _opt(pso, 32, sc3)
    checkpoint.load_optimizer_state(str(tmp_path / "plain"), opt3)
    assert sc3.get_scale() == 512.0 and int(sc3.growth_tracker.item()) == 0 and sc3.hyper()["growth_interval"] == 7


def test_fp16_tiny_unet_backs_off_from_overflow(pso):
    """The tiny SDXL fixture in fp16, r = 4, starting at S = 2^24: the first boundaries overflow and halve S without moving
    the parameters; the first finite boundary is bit-identical to an optimizer without a scaler given the same flat gradient
    and grad_scale = 1 / S."""
    from fixtures import micro_step, sdxl_unet
    from oracle import schedules
    L = pso.lora

    def build():
        torch.manual_seed(0)
        cfg = sdxl_unet.tiny_config()
        unet = sdxl_unet.UNet2DConditionModel(cfg).to(device="cuda", dtype=torch.float16)
        for w in L.add_adapter(unet, L.LoraConfig(r=4, lora_alpha=4)):
            torch.nn.init.normal_(w.lora_B["default"].weight, std=0.02)
        return cfg, unet

    cfg, unet = build()
    _, twin = build()
    sc = _scaler(pso, 2.0 ** 24)
    opt = L.FusedLoRAOptimizer(unet, **HYPER, grad_scaler=sc)
    ref = L.FusedLoRAOptimizer(twin, **HYPER)
    sched = schedules.turbo_scheduler(4)
    batch = micro_step.synth_batch(2, 64, cfg.cross_attention_dim, 32, 5, sched.sigmas)
    batch = {k: (v.cuda().half() if v.is_floating_point() and k not in ("human_prefer", "time_ids") else v.cuda())
             for k, v in batch.items()}

    def micro():
        ts = batch["timesteps"]
        p0 = micro_step._unet_call(unet, batch["input_latents_0"], ts, batch)
        p1 = micro_step._unet_call(unet, batch["input_latents_1"], ts, batch)
        L.disable_adapters(unet)
        with torch.no_grad():
            r0 = micro_step._unet_call(unet, batch["input_latents_0"], ts, batch)
            r1 = micro_step._unet_call(unet, batch["input_latents_1"], ts, batch)
        L.enable_adapters(unet)
        assert all(bool(torch.isfinite(t).all()) for t in (p0, p1, r0, r1)), "the fp16 forward overflowed"
        loss = pso.pso_pair_loss(p0, p1, r0, r1, batch["latents_0"], batch["latents_1"], batch["next_latents_0"],
                                 batch["next_latents_1"], ts, ts, batch["human_prefer"], scheduler=sched, grad_scaler=sc)
        sc.scale(loss).backward()
        return loss

    overflows = 0
    for b in range(16):
        S = sc.get_scale()
        loss = micro()
        assert torch.isfinite(loss).item()
        grad = opt.bucket.flat.clone()
        before = opt.flat_param.clone()
        ref.bucket.flat.copy_(grad)
        ref.grad_scale = float(ols.unscale_factor(np.float32(S)))
        opt.step()
        ref.step()
        if float(opt.found_inf) == 1.0:
            overflows += 1
            assert sc.get_scale() == S / 2 and torch.equal(opt.flat_param, before) and not bool(torch.isfinite(grad).all())
            assert torch.equal(ref.flat_param, before)
            continue
        assert overflows > 0, "S = 2^24 did not overflow the fp16 backward"
        assert torch.equal(opt.flat_param, ref.flat_param) and torch.equal(opt.exp_avg, ref.exp_avg)
        assert not torch.equal(opt.flat_param, before) and int(opt.step_dev.item()) == 1
        break
    else:
        pytest.fail("no finite boundary within 16 back-offs")
    print(f"fp16 tiny UNet: {overflows} overflowed boundaries, first finite update at S = {sc.get_scale():g}")


# ----------------------------------------------------------------------------------------------- two ranks
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_ranks_skip_together_and_hold_one_scale(built_lib):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(ROOT, "tests", "_loss_scaler_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-3000:] + "\n" + r.stderr[-6000:]
    assert "loss scaler exchange ok" in r.stdout

"""FusedLoRAOptimizer(optim_bits=8) -- psob200_flat_adamw8_step, bitsandbytes' blockwise 8-bit AdamW on the flat LoRA
buffers -- bit for bit against the restated oracle (oracle/optim8bit.py), against fp32 torch.optim.AdamW over 50 steps, and
through the overflow skip, checkpoint resume, CUDA-graph replay, padded operand copies and the fused two-GPU exchange."""
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import optim8bit as o8

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HYPER = dict(lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2, max_grad_norm=1.0)


@pytest.fixture(scope="module")
def L(built_lib):
    from pairwise_sample_optimization_b200 import lora
    return lora


def _model(L, r, seed=3, ragged=False):
    torch.manual_seed(seed)
    if ragged:  # matrices whose sizes are not multiples of 8 (scalar tails, padding behind them)
        m = torch.nn.ModuleDict({"to_q": torch.nn.Linear(100, 36, bias=False), "to_k": torch.nn.Linear(100, 36, bias=False),
                                 "to_v": torch.nn.Linear(52, 36, bias=False)})
    else:
        from tests.test_gpu_lora import _Attention
        m = _Attention(640, 2048, 10, 64)
    m = m.to(device="cuda", dtype=torch.bfloat16)
    wrapped = L.add_adapter(m, L.LoraConfig(r=r, lora_alpha=r))
    for w in wrapped:
        torch.nn.init.normal_(w.lora_B["default"].weight, std=0.05)
    return m, wrapped


def _opt8(L, r=8, seed=3, ragged=False, **kw):
    m, wrapped = _model(L, r, seed, ragged)
    return m, wrapped, L.FusedLoRAOptimizer(m, **HYPER, optim_bits=8, **kw)


def _state(opt):
    return {k: getattr(opt, k).cpu().numpy().copy() for k in ("code1", "code2", "absmax1", "absmax2", "exp_avg32",
                                                              "exp_avg_sq32", "qmap1", "qmap2")}


def _grads(n, k, seed=5, big_first=True):
    g = torch.Generator().manual_seed(seed)
    return [torch.randn(n, generator=g) * (3.0 if (i == 0 and big_first) else 1e-3) for i in range(k)]


@pytest.mark.parametrize("r,block_size,ragged", [(8, 256, False), (4, 256, False), (8, 2048, False), (4, 2048, False),
                                                 (5, 256, True), (5, 2048, True)])
def test_bitwise_against_the_oracle(L, r, block_size, ragged):
    """Five boundaries (the first one clips): codes, absmax, parameters, compact fp32 moments and operand copies are
    identical to the oracle's, which takes the kernel's reported norm for the clip coefficient."""
    _, _, opt = _opt8(L, r, ragged=ragged, block_size=block_size, min_8bit_size=200 if ragged else 4096)
    if r == 4:
        assert opt.chunks32.shape[0] > 0 and opt.blocks8.shape[0] > 0  # both classes present
    if ragged:
        assert bool((opt.blocks8[:, 1] % 8 != 0).any()) and bool((opt.chunks32[:, 1] % 8 != 0).any())
    blocks8, chunks32 = opt.blocks8.cpu().numpy(), opt.chunks32.cpu().numpy()
    st, p = _state(opt), opt.flat_param.cpu().numpy().copy()
    for t, grad in enumerate(_grads(opt.flat_param.numel(), 5), start=1):
        opt.bucket.flat.copy_(grad)
        norm = opt.step().item()
        if t == 1:
            assert norm > HYPER["max_grad_norm"]
        p, st = o8.adamw8_step(st, p, grad.numpy(), blocks8, chunks32, norm, t, HYPER["lr"], *HYPER["betas"], HYPER["eps"],
                               HYPER["weight_decay"], HYPER["max_grad_norm"])
        got = _state(opt)
        for k in st:
            assert np.array_equal(got[k], st[k]), f"step {t}: {k} differs from the oracle"
        assert np.array_equal(opt.flat_param.cpu().numpy(), p), f"step {t}: parameters differ from the oracle"
        assert torch.equal(opt.flat_operand.cpu(), torch.from_numpy(p).to(torch.bfloat16))
        assert float(opt.bucket.flat.abs().max()) == 0.0 and float(opt.found_inf) == 0.0 and int(opt.step_dev) == t
    # dequantized_moments() is qmap[code] * absmax on the 8-bit blocks and the compact moments elsewhere
    m, v = opt.dequantized_moments()
    blk, pos, _ = o8.table_positions(blocks8)
    assert np.array_equal(m.cpu().numpy()[pos], st["qmap1"][st["code1"][pos]] * st["absmax1"][blk])
    assert np.array_equal(v.cpu().numpy()[pos], st["qmap2"][st["code2"][pos]] * st["absmax2"][blk])
    if chunks32.shape[0]:
        _, pos, cpos = o8.table_positions(chunks32)
        assert np.array_equal(m.cpu().numpy()[pos], st["exp_avg32"][cpos])


# ||p_8bit - p_fp32|| / ||p_fp32 - p_0|| after 50 steps, measured at 1.622e-2 (B200, this seed); the bound leaves 3x margin
TRACKING_MEASURED = 1.622e-2


def test_tracks_fp32_adamw_over_50_steps(L):
    attn, _, opt = _opt8(L, 8)
    params = L.lora_parameters(attn)
    p0 = [p.detach().clone() for p in params]
    ref = [p.detach().clone().requires_grad_(True) for p in params]
    ref_opt = torch.optim.AdamW(ref, lr=HYPER["lr"], betas=HYPER["betas"], eps=HYPER["eps"], weight_decay=HYPER["weight_decay"])
    g = torch.Generator().manual_seed(7)
    drift = [torch.randn(p.shape, generator=g).cuda() * 0.01 for p in params]  # a consistent direction + noise
    for _ in range(50):
        for p, q, d in zip(params, ref, drift):
            grad = d + torch.randn(p.shape, generator=g).cuda() * 0.01
            p.grad.copy_(grad)
            q.grad = grad.clone()
        torch.nn.utils.clip_grad_norm_(ref, HYPER["max_grad_norm"])
        ref_opt.step()
        opt.step()
    dist = torch.sqrt(sum(((p.detach() - q.detach()) ** 2).sum() for p, q in zip(params, ref))).item()
    size = torch.sqrt(sum(((q.detach() - a) ** 2).sum() for q, a in zip(ref, p0))).item()
    print(f"8-bit vs fp32 AdamW after 50 steps: relative parameter distance {dist / size:.3e}")
    assert dist / size <= 3 * TRACKING_MEASURED


def test_overflow_skips_the_update(L):
    _, _, opt = _opt8(L, 4)
    _, _, ref = _opt8(L, 4)
    grads = _grads(opt.flat_param.numel(), 2, big_first=False)
    for o in (opt, ref):
        o.bucket.flat.copy_(grads[0])
        o.step()
    before = (_state(opt), opt.flat_param.clone(), opt.flat_operand.clone())
    for bad in (float("inf"), float("nan")):
        opt.bucket.flat.copy_(grads[1])
        opt.bucket.flat[1234] = bad
        norm = opt.step()
        assert not torch.isfinite(norm).item() and float(opt.found_inf) == 1.0 and int(opt.step_dev.item()) == 1
        assert float(opt.bucket.flat.abs().max()) == 0.0
        got = _state(opt)
        assert all(np.array_equal(got[k], before[0][k]) for k in got)
        assert torch.equal(opt.flat_param, before[1]) and torch.equal(opt.flat_operand, before[2])
    for o in (opt, ref):  # the next finite step is the second update of both runs
        o.bucket.flat.copy_(grads[1])
        o.step()
    assert float(opt.found_inf) == 0.0 and torch.equal(opt.flat_param, ref.flat_param)
    assert all(np.array_equal(a, b) for a, b in zip(_state(opt).values(), _state(ref).values()))


def test_checkpoint_resume_is_bit_identical_and_other_layouts_are_refused(L, tmp_path):
    from pairwise_sample_optimization_b200 import _lib, checkpoint
    attn, _, opt = _opt8(L, 4)
    grads = _grads(opt.flat_param.numel(), 4, big_first=False)
    for k in range(2):
        opt.bucket.flat.copy_(grads[k])
        opt.step()
    checkpoint.save_state(str(tmp_path), attn, opt)
    from safetensors import safe_open
    with safe_open(os.path.join(str(tmp_path), checkpoint.OPTIMIZER_NAME), framework="pt") as f:
        meta, keys = f.metadata(), set(f.keys())
        assert f.get_tensor("code1").dtype == torch.uint8
    assert meta["optim_bits"] == "8" and meta["block_size"] == "256" and meta["min_8bit_size"] == "4096"
    assert keys == {"flat_param", "code1", "code2", "absmax1", "absmax2", "exp_avg32", "exp_avg_sq32", "qmap1", "qmap2"}
    attn2, wrapped2, opt2 = _opt8(L, 4, seed=99)
    assert not torch.equal(opt2.flat_param, opt.flat_param)
    checkpoint.load_state(str(tmp_path), attn2, opt2)
    assert int(opt2.step_dev.item()) == 2
    for m in wrapped2:
        for which, lin in (("a", m.lora_A["default"]), ("b", m.lora_B["default"])):
            assert torch.equal(m._operand(which, torch.bfloat16), lin.weight.detach().to(torch.bfloat16))
    for k in (2, 3):
        for o in (opt, opt2):
            o.bucket.flat.copy_(grads[k])
            o.step()
    assert torch.equal(opt2.flat_param, opt.flat_param)
    assert all(np.array_equal(a, b) for a, b in zip(_state(opt).values(), _state(opt2).values()))
    # the other mode, another block layout, another flat layout: refused with a clear message
    a32, _ = _model(L, 4)
    opt32 = L.FusedLoRAOptimizer(a32, **HYPER)
    with pytest.raises(_lib.Psob200Error, match="optim_bits"):
        checkpoint.load_optimizer_state(str(tmp_path), opt32)
    checkpoint.save_optimizer_state(str(tmp_path / "fp32"), opt32)
    with pytest.raises(_lib.Psob200Error, match="optim_bits"):
        checkpoint.load_optimizer_state(str(tmp_path / "fp32"), opt2)
    _, _, opt_bs = _opt8(L, 4, block_size=2048)
    with pytest.raises(_lib.Psob200Error, match="block_size"):
        checkpoint.load_optimizer_state(str(tmp_path), opt_bs)
    _, _, opt_r = _opt8(L, 8)
    with pytest.raises(_lib.Psob200Error, match="layout"):
        checkpoint.load_optimizer_state(str(tmp_path), opt_r)


def test_cuda_graph_replay_equals_the_eager_step(L):
    _, _, eager = _opt8(L, 8)
    _, _, graphed = _opt8(L, 8)
    grads = [g.cuda() for g in _grads(eager.flat_param.numel(), 4)]
    for o in (eager, graphed):
        o.bucket.flat.copy_(grads[0])
        o.step()
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        graphed.step()
    for k in (1, 2, 3):
        graphed.bucket.flat.copy_(grads[k])
        graph.replay()
        eager.bucket.flat.copy_(grads[k])
        eager.step()
        torch.cuda.synchronize()
        assert torch.equal(graphed.flat_param, eager.flat_param) and torch.equal(graphed.flat_operand, eager.flat_operand)
        assert all(np.array_equal(a, b) for a, b in zip(_state(graphed).values(), _state(eager).values()))
        assert int(graphed.step_dev.item()) == k + 1


def test_padded_operand_copies_follow_the_parameters(L):
    """r = 4 with fuse_attention_projections: the stacked k / v group keeps padded private operands ([G * 8, K], zero rows
    behind each projection's 4), q / out keep padded per-layer copies; the 8-bit boundary refreshes all of them."""
    from tests.test_gpu_lora import _Attention
    dtype = torch.bfloat16
    torch.manual_seed(3)
    attn = _Attention(640, 2048, 10, 64).to(device="cuda", dtype=dtype)
    wrapped = L.add_adapter(attn, L.LoraConfig(r=4, lora_alpha=4))
    for m in wrapped:
        torch.nn.init.normal_(m.lora_B["default"].weight, std=0.05)
    assert L.fuse_attention_projections(attn) == 1
    opt = L.FusedLoRAOptimizer(attn, **HYPER, optim_bits=8)
    assert opt.blocks8.shape[0] > 0 and opt.chunks32.shape[0] > 0
    grp = L.projection_groups(attn)[0]
    grp.refresh_operands()
    opt.bucket.flat.copy_(_grads(opt.flat_param.numel(), 1)[0].cuda())
    opt.step()
    rs = grp.r_stride
    sa = grp.stacked_operand("a", dtype)
    for g, lay in enumerate(grp.layers):
        assert torch.equal(sa[g * rs:g * rs + 4], lay.lora_A["default"].weight.detach().to(dtype))
        assert float(sa[g * rs + 4:(g + 1) * rs].abs().max()) == 0.0
        n = lay.out_features
        assert torch.equal(grp.stacked_operand("b", dtype)[g * n:(g + 1) * n], lay.lora_B["default"].weight.detach().to(dtype))
    for m in wrapped:
        for which, lin in (("a", m.lora_A["default"]), ("b", m.lora_B["default"])):
            assert torch.equal(m._operand(which, dtype), lin.weight.detach().to(dtype))


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_ranks_hold_identical_8bit_state_with_the_fused_exchange(built_lib):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(_free_port()), os.path.join(ROOT, "tests", "_optim8bit_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-3000:] + "\n" + r.stderr[-6000:]
    assert "8-bit exchange ok" in r.stdout

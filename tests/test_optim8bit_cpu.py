"""CPU: the host side of the 8-bit AdamW state (``FusedLoRAOptimizer(optim_bits=8)``): the quantisation maps, the block
tables of the SDXL flat layout, the oracle's quantiser, and the argument checks of psob200_flat_adamw8_step."""
import ctypes as C

import numpy as np
import pytest
import torch

from fixtures import sdxl_unet
from oracle import optim8bit as o8


def test_dynamic_maps_facts_and_host_builder_matches_the_oracle():
    from pairwise_sample_optimization_b200 import lora
    s, u = lora.dynamic_quant_map(True), lora.dynamic_quant_map(False)
    assert s.dtype == torch.float32 and u.dtype == torch.float32
    assert np.array_equal(s.numpy(), o8.create_dynamic_map(True)) and np.array_equal(u.numpy(), o8.create_dynamic_map(False))
    for q in (s, u):
        assert q.numel() == 256 and torch.unique(q).numel() == 256 and bool((q[1:] > q[:-1]).all())
    assert s[127].item() == 0.0 and s[0].item() == np.float32(-0.99296874) and s[255].item() == 1.0
    assert abs(s[s > 0].min().item() - 5.5e-7) < 1e-12
    assert u[0].item() == 0.0 and u[255].item() == 1.0


def _sdxl_layout(r):
    """numels and 8-aligned flat offsets of the 1 120 adapter matrices of the SDXL UNet at rank r (A = [r, in], B = [out, r])."""
    with torch.device("meta"):
        unet = sdxl_unet.UNet2DConditionModel(sdxl_unet.sdxl_config())
    numels, offsets, off = [], [], 0
    for name, m in unet.named_modules():
        if isinstance(m, torch.nn.Linear) and name.endswith((".to_q", ".to_k", ".to_v", ".to_out.0")):
            for n in (r * m.in_features, m.out_features * r):
                numels.append(n)
                offsets.append(off)
                off += (n + 7) // 8 * 8
    return numels, offsets


@pytest.mark.parametrize("r", [4, 64])
@pytest.mark.parametrize("block_size", [256, 2048])
def test_block_tables_of_the_sdxl_layout(r, block_size):
    from pairwise_sample_optimization_b200 import lora
    numels, offsets = _sdxl_layout(r)
    assert len(numels) == 1120 and sum(numels) == 1451520 * r
    blocks8, chunks32, n32 = lora.blockwise_layout(numels, offsets, block_size, 4096)
    small = [(n, off) for n, off in zip(numels, offsets) if n < 4096]
    big = [(n, off) for n, off in zip(numels, offsets) if n >= 4096]
    if r == 4:  # the 640-wide A [4, 640] and B [640, 4] (2 560 elements) keep fp32 moments
        assert small and all(n == 2560 for n, _ in small)
    else:
        assert not small and chunks32.shape[0] == 0 and n32 == 0
    assert blocks8.shape[0] == sum(-(-n // block_size) for n, _ in big)
    assert int(blocks8[:, 1].sum()) == sum(n for n, _ in big)
    assert int(blocks8[:, 1].max()) <= block_size and bool((blocks8[:, 0] % 8 == 0).all())
    short = blocks8[blocks8[:, 1] < block_size]
    assert short.shape[0] == sum(1 for n, _ in big if n % block_size)
    if r == 4 and block_size == 2048:  # 1280-wide: 5 120 = 2 x 2048 + 1024
        assert short.shape[0] > 0 and 1024 in short[:, 1].tolist()
    # every 8-bit matrix is tiled from its own offset, block after block
    starts = {off for _, off in big}
    firsts = blocks8[:, 0].tolist()
    assert starts <= set(firsts)
    if small:
        assert int(chunks32[:, 1].sum()) == sum(n for n, _ in small) and n32 == sum((n + 7) // 8 * 8 for n, _ in small)
        assert bool((chunks32[:, 2] % 8 == 0).all()) and int(chunks32[:, 1].max()) <= block_size


def test_block_tables_of_an_odd_layout():
    from pairwise_sample_optimization_b200 import lora
    blocks8, chunks32, n32 = lora.blockwise_layout([5000, 100, 4096, 600], [0, 5000, 5104, 9200], 256, 4096)
    assert blocks8.tolist()[:2] == [[0, 256], [256, 256]] and blocks8.tolist()[19] == [4864, 136]
    assert blocks8.tolist()[20] == [5104, 256] and blocks8.shape[0] == 20 + 16
    assert chunks32.tolist() == [[5000, 100, 0], [9200, 256, 104], [9456, 256, 360], [9712, 88, 616]] and n32 == 704
    with pytest.raises(ValueError):
        lora.blockwise_layout([10], [4])


def test_oracle_quantise_round_trip_and_sign_rule():
    rng = np.random.default_rng(0)
    for signed in (True, False):
        q = o8.create_dynamic_map(signed)
        lo = -1.0 if signed else 0.0
        # values across all decades, both signs
        x = (rng.uniform(lo, 1.0, 20000) * 10.0 ** rng.integers(-7, 1, 20000)).astype(np.float32)
        x = np.clip(x, q[0], q[-1])
        m = x if signed else None
        c = o8.quantize(x, q, m)
        d = q[c]
        i = np.clip(np.searchsorted(q, x, side="right") - 1, 0, 254)  # x in [q[i], q[i+1]]
        gap = q[i + 1] - q[i]
        moved = np.zeros_like(x, dtype=bool)
        if signed:  # the sign rule may move a tiny value by one code, never across zero
            assert not np.any(np.signbit(d) != np.signbit(x))
            moved = c != o8.quantize(x, q)
            assert np.all(np.abs(x[moved]) < 5.5e-7)
        assert np.all(np.abs(d - x)[~moved] <= 0.5 * gap[~moved])
        # absmax = 0 gives x = 0, the code of 0.0
        zero = o8.quantize(np.zeros(3, np.float32), q, np.zeros(3, np.float32) if signed else None)
        assert np.all(q[zero] == 0.0) and zero[0] == (127 if signed else 0)
    # a tiny negative momentum stays negative instead of rounding to +0
    q1 = o8.create_dynamic_map(True)
    assert o8.quantize(np.array([-1e-7], np.float32), q1, np.array([-1e-7], np.float32))[0] == 126


def test_optimizer_arguments_are_checked_before_any_device_work():
    from pairwise_sample_optimization_b200 import lora
    net = torch.nn.Linear(8, 8)
    with pytest.raises(ValueError, match="optim_bits"):
        lora.FusedLoRAOptimizer(net, optim_bits=4)
    with pytest.raises(ValueError, match="block_size"):
        lora.FusedLoRAOptimizer(net, optim_bits=8, block_size=512)


def test_adamw8_entry_argument_validation_without_gpu(built_lib):
    from pairwise_sample_optimization_b200 import _lib
    lib = _lib.lib()
    assert lib.psob200_flat_adamw8_step(None, None) == -1
    o = _lib.FlatAdamw8Args()
    o.param = o.grad = o.workspace = o.code1 = o.code2 = o.absmax1 = o.absmax2 = o.map1 = o.map2 = o.blocks8 = 4096
    o.n, o.step, o.n_blocks8, o.block_size = 4096, 1, 16, 256
    o.n_sumsq_parts = 2  # pieces announced but no pointer to them
    assert lib.psob200_flat_adamw8_step(C.byref(o), None) == -1
    o.n_sumsq_parts = 0
    o.n_chunks32 = 1  # fp32-class ranges without their table or state
    assert lib.psob200_flat_adamw8_step(C.byref(o), None) == -1
    o.n_chunks32 = 0
    o.block_size = 512
    assert lib.psob200_flat_adamw8_step(C.byref(o), None) == -5  # 256 or 2048 only
    o.block_size = 2048
    o.code2 = 4096 + 8
    assert lib.psob200_flat_adamw8_step(C.byref(o), None) == -3  # code arrays 16-byte aligned
    o.code2, o.param = 4096, 4100
    assert lib.psob200_flat_adamw8_step(C.byref(o), None) == -3

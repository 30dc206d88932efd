"""GPU parity of the fused norms (psob200_layer_norm_* / psob200_group_norm_*): forward and input gradient against torch in
fp64 on the same inputs, never worse than the stock op by more than 1 ulp; autocast; the stock fallback of the patched
modules; determinism and CUDA-graph replay; the tiny and the full SDXL fixture end to end."""
import pytest
import torch
import torch.nn.functional as F

from fixtures import micro_step, sdxl_unet
from tests import _util as U

pytestmark = pytest.mark.gpu

EPS_ULP = {torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -11, torch.float32: 2.0 ** -24}  # half an ulp, relative
# fp32 statistics and exp carry relative errors of ~1e-6: an exact result that close to a rounding boundary of the 16-bit
# type rounds either way.  Measured well below 1 %; none may be off by more than 1 ulp.
MISMATCH = 0.02


@pytest.fixture(scope="module")
def nm(built_lib):
    from pairwise_sample_optimization_b200 import norms
    return norms


def _inputs(shape, dtype, seed, affine, params_dtype=None):
    g = torch.Generator().manual_seed(seed)
    x = (torch.randn(*shape, generator=g) * 1.5 + 0.7).to(dtype).cuda()
    c = shape[1] if len(shape) == 4 else shape[-1]
    w = b = None
    if affine:
        pd = params_dtype or dtype
        w = (1.0 + 0.3 * torch.randn(c, generator=g)).to(pd).cuda()
        b = (0.2 * torch.randn(c, generator=g)).to(pd).cuda()
    return x, w, b, g


def _check(got, want, stock, dtype):
    """fp32: 1e-5 relative max (BASELINE's north star); 16-bit: correctly rounded up to 1 ulp almost everywhere.  And the
    fused error is never worse than the stock op's on the same inputs by more than 1 ulp at the largest magnitude."""
    want = want.cpu()
    if dtype == torch.float32 and got.dtype == torch.float32:
        assert U.rel_max(got, want) <= 1e-5
    else:
        U.assert_rounded_equal(got, want, got.dtype, max_mismatch_frac=MISMATCH)
    err = (got.double().cpu() - want.cpu()).abs().max().item()
    err_stock = (stock.double().cpu() - want.cpu()).abs().max().item()
    assert err <= err_stock + 2 * EPS_ULP[got.dtype] * want.abs().max().item(), (err, err_stock)


def _truth_and_stock(fn, x, dy, *args):
    """fn in fp64 (truth) and in the input's own type (stock kernels): outputs and input gradients."""
    x64 = x.detach().double().requires_grad_(True)
    y64 = fn(x64, *[a.double() if torch.is_tensor(a) else a for a in args])
    y64.backward(dy.double())
    xs = x.detach().clone().requires_grad_(True)
    ys = fn(xs, *args)
    ys.backward(dy.to(ys.dtype))
    return y64.detach(), x64.grad, ys.detach(), xs.grad


@pytest.mark.parametrize("dtype", ["bf16", "fp16", "fp32"])
@pytest.mark.parametrize("affine", [True, False])
@pytest.mark.parametrize("shape", [(2 * 4096, 640), (2 * 1024, 1280), (3, 77, 32), (5, 64), (1001, 320)])
def test_layer_norm(nm, dtype, affine, shape):
    dt = U.DT[dtype]
    x, w, b, g = _inputs(shape, dt, 1, affine)
    dy = torch.randn(*shape, generator=g).to(dt).cuda()
    xf = x.clone().requires_grad_(True)
    y = nm.layer_norm(xf, w, b, 1e-5)
    y.backward(dy)
    assert y.dtype == dt and xf.grad.dtype == dt
    fn = lambda t, ww, bb: F.layer_norm(t, (shape[-1],), ww, bb, 1e-5)
    y64, dx64, ys, dxs = _truth_and_stock(fn, x, dy, w, b)
    _check(y, y64, ys, dt)
    _check(xf.grad, dx64, dxs, dt)


def _gn_ref(x, ca, G, w, b, eps, silu):
    if ca is not None:
        x = (x + ca[:, :, None, None]).to(x.dtype)  # the stock add rounds to the input type
    y = F.group_norm(x, G, w, b, eps)
    return F.silu(y) if silu else y


GN_SHAPES = [((1, 960, 128, 128), 32), ((2, 640, 64, 64), 32), ((2, 64, 16, 16), 32), ((2, 32, 7, 9), 32),
             ((3, 12, 5, 5), 4), ((1, 8, 1, 1), 2)]


@pytest.mark.parametrize("dtype", ["bf16", "fp16", "fp32"])
@pytest.mark.parametrize("mode", ["plain", "silu", "silu_add"])
@pytest.mark.parametrize("shape,G", GN_SHAPES)
def test_group_norm(nm, dtype, mode, shape, G):
    dt = U.DT[dtype]
    affine = shape[1] != 12  # one shape without the affine
    x, w, b, g = _inputs(shape, dt, 2, affine)
    silu = mode != "plain"
    ca = (torch.randn(shape[0], shape[1], generator=g) * 0.5).to(dt).cuda() if mode == "silu_add" else None
    dy = torch.randn(*shape, generator=g).to(dt).cuda()
    xf = x.clone().requires_grad_(True)
    y = nm.group_norm(xf, G, w, b, 1e-5, silu=silu, channel_add=ca)
    y.backward(dy)
    assert y.dtype == dt and xf.grad.dtype == dt
    # truth: the rounded sum x + channel_add is the normalised input in both; fp64 from there on
    xs_in = x if ca is None else (x + ca[:, :, None, None]).to(dt)
    fn = lambda t, ww, bb: _gn_ref(t, None, G, ww, bb, 1e-5, silu)
    y64, dx64, ys, dxs = _truth_and_stock(fn, xs_in, dy, w, b)
    _check(y, y64, ys, dt)
    _check(xf.grad, dx64, dxs, dt)


def test_fp32_params_with_16bit_input_and_errors(nm):
    from pairwise_sample_optimization_b200 import _lib
    x, w, b, g = _inputs((4, 64, 8, 8), torch.bfloat16, 3, True, params_dtype=torch.float32)
    y = nm.group_norm(x, 32, w, b, 1e-6)
    want = F.group_norm(x.double(), 32, w.double(), b.double(), 1e-6)
    U.assert_rounded_equal(y, want.cpu(), torch.bfloat16, max_mismatch_frac=MISMATCH)
    with pytest.raises(_lib.Psob200Error):
        nm.group_norm(x, 7, w, b)  # 64 channels in 7 groups
    with pytest.raises(_lib.Psob200Error):
        nm.layer_norm(torch.randn(4, 20, device="cuda"))  # width not a multiple of 8


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_autocast_patched_modules(nm, dtype):
    torch.manual_seed(0)
    mods = torch.nn.ModuleList([torch.nn.LayerNorm(640), torch.nn.GroupNorm(32, 320)]).cuda().requires_grad_(False)
    stock = [torch.nn.LayerNorm(640), torch.nn.GroupNorm(32, 320)]
    for s, m in zip(stock, mods):
        s.load_state_dict(m.state_dict())
    stock = torch.nn.ModuleList(stock).cuda().requires_grad_(False)
    assert nm.install_fused_norms(mods) == {"layer_norm": 1, "group_norm": 1, "resnet_block": 0}
    for i, shape in enumerate([(2, 256, 640), (2, 320, 16, 16)]):
        x = torch.randn(*shape, device="cuda").to(dtype)
        with torch.autocast("cuda", dtype):
            got, want = mods[i](x), stock[i](x)
        assert got.dtype == want.dtype == torch.float32
        assert U.rel_max(got, want) <= 1e-5


def test_trainable_weight_takes_the_stock_path(nm):
    torch.manual_seed(0)
    for make, shape in ((lambda: torch.nn.LayerNorm(64), (3, 10, 64)), (lambda: torch.nn.GroupNorm(4, 16), (2, 16, 5, 5))):
        stock, fused = make().cuda().bfloat16(), make().cuda().bfloat16()
        fused.load_state_dict(stock.state_dict())
        nm.install_fused_norms(fused)
        x = torch.randn(*shape, device="cuda").bfloat16()
        xs, xf = x.clone().requires_grad_(True), x.clone().requires_grad_(True)
        ys, yf = stock(xs), fused(xf)
        ys.float().square().sum().backward()
        yf.float().square().sum().backward()
        assert torch.equal(ys, yf) and torch.equal(xs.grad, xf.grad)
        assert fused.weight.grad is not None and torch.equal(fused.weight.grad, stock.weight.grad)


def test_deterministic_and_graph_replay(nm):
    torch.manual_seed(0)
    x = torch.randn(2, 960, 64, 64, device="cuda").bfloat16()
    ca = torch.randn(2, 960, device="cuda").bfloat16()
    w, b = torch.randn(960, device="cuda").bfloat16(), torch.randn(960, device="cuda").bfloat16()
    xl = torch.randn(2 * 4096, 640, device="cuda").bfloat16()
    wl = torch.randn(640, device="cuda").bfloat16()
    dy, dyl = torch.randn_like(x), torch.randn_like(xl)

    def run():
        xi, xli = x.clone().requires_grad_(True), xl.clone().requires_grad_(True)
        y = nm.group_norm(xi, 32, w, b, 1e-5, silu=True, channel_add=ca)
        yl = nm.layer_norm(xli, wl, None, 1e-5)
        torch.autograd.backward([y, yl], [dy, dyl])
        return [y.detach(), xi.grad, yl.detach(), xli.grad]

    first, second = run(), run()
    assert all(torch.equal(a, b_) for a, b_ in zip(first, second))
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        run()
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=side):
        static = run()
    graph.replay()
    torch.cuda.synchronize()
    assert all(torch.equal(a, b_) for a, b_ in zip(first, static))


def _lora_unet(cfg, r, seed=1234):
    from pairwise_sample_optimization_b200 import lora
    torch.manual_seed(seed)
    with torch.device("cuda"):
        unet = sdxl_unet.UNet2DConditionModel(cfg)
    unet = unet.to(torch.bfloat16).requires_grad_(False)
    wrapped = lora.add_adapter(unet, lora.LoraConfig(r=r, lora_alpha=r))
    for m in wrapped:
        torch.nn.init.normal_(m.lora_B["default"].weight, std=0.01)
    unet.set_attn_processor(lora.PSOAttnProcessor2_0())
    unet.train()
    return unet, wrapped


def _single_rounding_stock(unet):
    """Stock torch computing what the fused ResNet path computes: GroupNorm (+ the rounded time-embedding add) and SiLU in
    fp32, ONE rounding to the activation type.  The plain stock lines round the norm's output before the SiLU; on the random
    SDXL fixture at B = 1 that second rounding alone moves the dmd128 loss by ~5 % (measured against the fused kernels: loss
    0.672 vs 0.642, gradient cosine 0.998, norm ratio 1.025), so plain stock is no yardstick for ulp-level agreement."""
    def patch(m):
        def gn_silu(x, n, t=None):
            if t is not None:
                x = x + t[:, :, None, None]
            return F.silu(F.group_norm(x.float(), n.num_groups, n.weight.float(), n.bias.float(), n.eps)).to(x.dtype)

        def forward(x, temb):
            h = m.conv1(gn_silu(x, m.norm1))
            h = m.conv2(gn_silu(h, m.norm2, m.time_emb_proj(F.silu(temb))))
            return (x if m.conv_shortcut is None else m.conv_shortcut(x)) + h
        return forward
    for m in unet.modules():
        if type(m).__name__ == "ResnetBlock2D":
            m.forward = patch(m)


def _grads(layers):
    out = torch.cat([torch.cat([m.lora_A["default"].weight.grad.flatten(), m.lora_B["default"].weight.grad.flatten()])
                     for m in layers]).double().cpu()
    for m in layers:
        m.lora_A["default"].weight.grad = m.lora_B["default"].weight.grad = None
    return out


def test_tiny_fixture_forward_backward_matches_single_rounding_stock(nm):
    cfg = sdxl_unet.tiny_config()
    unet, wrapped = _lora_unet(cfg, 4)
    pooled = cfg.projection_class_embeddings_input_dim - 6 * cfg.addition_time_embed_dim
    d = {k: v.cuda() for k, v in micro_step.synth_batch(2, 32, cfg.cross_attention_dim, pooled, 5, None,
                                                        dtype=torch.bfloat16, kind="dmd").items()}

    def fwd_bwd():
        out = micro_step._unet_call(unet, d["input_latents_0"], d["timesteps"], d)
        out.float().square().mean().backward()
        return out.detach().float(), _grads(wrapped)

    _single_rounding_stock(unet)
    y_s, g_s = fwd_bwd()
    assert nm.install_fused_norms(unet) == {"layer_norm": 36, "group_norm": 31, "resnet_block": 12}
    y_f, g_f = fwd_bwd()
    assert U.rel_max(y_f, y_s) <= 3e-2  # bf16 activations through 12 ResNet blocks and 12 transformer blocks
    cos = (torch.dot(g_s, g_f) / (g_s.norm() * g_f.norm())).item()
    assert g_s.abs().max() > 0 and cos >= 0.999, cos


def test_full_sdxl_dmd128_step_fused_vs_single_rounding_stock_and_graph_replay(nm):
    import pairwise_sample_optimization_b200 as pso
    from oracle import schedules
    from pairwise_sample_optimization_b200 import lora
    cfg = sdxl_unet.sdxl_config()
    unet, _ = _lora_unet(cfg, 64)
    opt = lora.FusedLoRAOptimizer(unet)
    sched = schedules.dmd_scheduler()
    pooled = cfg.projection_class_embeddings_input_dim - 6 * cfg.addition_time_embed_dim
    host = micro_step.synth_batch(1, 128, cfg.cross_attention_dim, pooled, 100, None, dtype=torch.bfloat16, kind="dmd")
    d = micro_step.batched_view({k: v.cuda() for k, v in host.items()})
    kw = dict(beta=50.0, eps=0.1, kind="dmd")
    lora.set_wgrad_stream(False)
    lora.set_deterministic_wgrad(True)
    try:
        def eager():
            opt.bucket.zero_()
            loss = micro_step.product_micro_step_batched(pso, lora, unet, d, sched, **kw)
            torch.cuda.synchronize()
            return float(loss.item()), opt.bucket.flat.double().cpu().clone()

        _single_rounding_stock(unet)
        loss_s, g_s = eager()
        assert g_s.abs().max() > 0, "vacuous: every gradient is zero"
        assert nm.install_fused_norms(unet) == {"layer_norm": 210, "group_norm": 46, "resnet_block": 17}
        loss_f, g_f = eager()
        cos = (torch.dot(g_s, g_f) / (g_s.norm() * g_f.norm())).item()
        report = (loss_f, loss_s, cos, g_f.norm().item() / g_s.norm().item())
        # the bounds of the batched-versus-separate comparison (two bf16 evaluations of the same step)
        assert abs(loss_f - loss_s) <= 1e-2 * abs(loss_s), report
        assert cos >= 0.995 and abs(report[3] - 1.0) <= 2e-2, report
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            micro_step.product_micro_step_batched(pso, lora, unet, d, sched, **kw)
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            static_loss = micro_step.product_micro_step_batched(pso, lora, unet, d, sched, **kw)
        graph.replay()
        torch.cuda.synchronize()
        assert float(static_loss.item()) == loss_f, (float(static_loss.item()), loss_f)
    finally:
        lora.set_deterministic_wgrad(False)

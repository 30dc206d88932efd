"""Fused PSO losses (host side) -- the "new function whose body is the reference's inline code"
(SURVEY.md section 8b, boundary b2).

``pso_pair_loss`` replaces, verbatim in meaning, the four ``*_step_with_logprob`` calls + the
inline loss of one micro-step (train_online_pso_sdxl_turbo.py:810-850,
train_online_pso_sdxl_dmd2.py:812-854); ``pso_db_loss`` replaces
train_pso_sdxl_turbo_dreambooth.py:1847-1865 + 1881-1935.  Both launch ONE kernel that also
produces the gradient w.r.t. the policy predictions, which ``backward`` then hands to autograd.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib, amp, runtime


# ----------------------------------------------------------------------------- preference signs (a4)
def sample_compare(a: torch.Tensor, b: torch.Tensor, generator=None) -> torch.Tensor:
    """train_online_pso_sdxl_turbo.py:401-416: one random reward column per row;
    ``a <= b`` -> [-1, +1] (ties favour sample 1), else [+1, -1].  No host sync (the reference's
    boolean-mask assignment syncs)."""
    bs, num_rewards = a.shape
    idx = torch.randint(0, num_rewards, (bs,), device=a.device, generator=generator)
    pa = a.gather(1, idx[:, None]).squeeze(1)
    pb = b.gather(1, idx[:, None]).squeeze(1)
    # explicit masks like the reference's (a_dom = pa <= pb, b_dom = pb < pa): a NaN reward satisfies neither -> [0, 0]
    s = (pa <= pb).to(torch.float) - (pb < pa).to(torch.float)
    return torch.stack([-s, s], dim=1)


def compare(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """train_online_pso_sdxl_dmd2.py:420-434: Pareto dominance; ties / incomparable -> [0, 0]."""
    assert isinstance(a, torch.Tensor) and isinstance(b, torch.Tensor)
    if a.dim() == 1:
        a = a[..., None]
        b = b[..., None]
    a_dom = torch.logical_and(torch.all(a <= b, dim=1), torch.any(a < b, dim=1))
    b_dom = torch.logical_and(torch.all(b <= a, dim=1), torch.any(b < a, dim=1))
    s = a_dom.to(torch.float) - b_dom.to(torch.float)  # +1: sample 1 wins, -1: sample 0 wins, 0: tie
    return torch.stack([-s, s], dim=1)


# ----------------------------------------------------------------------------- online PSO
def _n(t):
    n = 1
    for s in t.shape[1:]:
        n *= int(s)
    return n


def _launch_loss(dev, name, scaler, *args):
    """The loss launch, through the ``_scaled`` entry point when a ``DeviceGradScaler`` is given."""
    if scaler is None:
        _lib.launch(dev, name, *args, _lib.current_stream(dev))
    else:
        s = amp.scaler_arg(scaler, dev)
        _lib.launch(dev, name + "_scaled", *args, C.byref(s), _lib.current_stream(dev))


def _apply_upstream(grads, grad_out, dev, scaler=None):
    """d loss was folded into the kernel as 1 (as S with a loss scaler); scale by autograd's upstream gradient (divided by
    S) on the device -- a no-op launch when that is exactly 1, e.g. after ``scaler.scale(loss).backward()``."""
    go = grad_out.detach().reshape(1).to(torch.float32)
    if scaler is not None:
        go = go / scaler.scale_tensor
    for g in grads:
        _lib.launch(dev, "psob200_scale_inplace_by_device_scalar", g.data_ptr(), g.numel(), _lib.dtype_code(g),
                                                               go.data_ptr(), _lib.current_stream(dev))


class _OnlinePsoLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pred0, pred1, ref0, ref1, x0, x1, xn0, xn1, ts0, ts1, tsp0, tsp1, coef0, coef1, h, sched,
                beta, eps, loss_scale, want_stats, tune, scaler):
        dev = _lib.require_cuda(pred0, pred1, ref0, ref1, x0, x1, xn0, xn1, h)
        B, n = pred0.shape[0], _n(pred0)
        a = _lib.OnlinePsoArgs()
        keep = []
        if pred1.dtype != pred0.dtype or ref0.dtype != pred0.dtype or ref1.dtype != pred0.dtype:
            raise _lib.Psob200Error("policy and reference predictions must share one dtype")
        lat_dtype = x0.dtype
        for k, (p, r, x, xn) in enumerate(((pred0, ref0, x0, xn0), (pred1, ref1, x1, xn1))):
            if p.shape[0] != B or _n(p) != n or _n(r) != n or _n(x) != n or _n(xn) != n:
                raise _lib.Psob200Error("pso_pair_loss: all eight tensors must have the same [B, ...] shape")
            x = x if x.dtype == lat_dtype else x.to(lat_dtype)
            xn = xn if xn.dtype == lat_dtype else xn.to(lat_dtype)
            for name, t in (("pred", p), ("ref", r), ("sample", x), ("next", xn)):
                tt, st = _lib.rows(t, n)
                keep.append(tt)
                getattr(a, name)[k] = tt.data_ptr()
                getattr(a, "stride_" + name)[k] = st
        for k, (ts, tsp, cf) in enumerate(((ts0, tsp0, coef0), (ts1, tsp1, coef1))):
            a.ts[k] = ts.data_ptr() if ts is not None else None
            a.ts_prev[k] = tsp.data_ptr() if tsp is not None else None
            a.coef[k] = cf.data_ptr() if cf is not None else None
        hp = h.detach().to(device=dev, dtype=torch.float32).contiguous()
        if hp.shape != (B, 2):
            raise _lib.Psob200Error(f"human_prefer must be [B,2], got {tuple(hp.shape)}")
        a.human_prefer = hp.data_ptr()
        grad0 = torch.empty(pred0.shape, dtype=pred0.dtype, device=dev)
        grad1 = torch.empty(pred1.shape, dtype=pred1.dtype, device=dev)
        loss = torch.empty((), dtype=torch.float32, device=dev)
        stats = torch.empty((B, 8), dtype=torch.float32, device=dev) if want_stats else None
        nbytes = _lib.lib().psob200_pair_loss_workspace_bytes(B)
        ws = runtime.workspace(dev, nbytes)
        a.grad[0], a.grad[1] = grad0.data_ptr(), grad1.data_ptr()
        a.loss = loss.data_ptr()
        a.stats = stats.data_ptr() if stats is not None else None
        a.status = runtime.status_word(dev).data_ptr()
        a.workspace, a.workspace_bytes = ws.data_ptr(), ws.numel()
        a.B, a.N = B, n
        a.pred_dtype, a.latent_dtype = _lib.dtype_code(pred0), _lib.dtype_code(keep[2])
        a.beta, a.eps, a.loss_scale = float(beta), float(eps), float(loss_scale)
        a.tune_threads, a.tune_cluster = tune
        _launch_loss(dev, "psob200_online_pso_loss_grad", scaler, sched.ref(), C.byref(a))
        ctx.save_for_backward(grad0, grad1)
        ctx.dev = dev
        ctx.scaler = scaler
        ctx.used = False
        if stats is not None:
            ctx.mark_non_differentiable(stats)
            return loss, stats
        return loss, None

    @staticmethod
    def backward(ctx, grad_loss, _grad_stats):
        if ctx.used:
            raise RuntimeError("pso_pair_loss: backward may run only once (its gradient buffers are consumed)")
        ctx.used = True
        grad0, grad1 = ctx.saved_tensors
        _apply_upstream((grad0, grad1), grad_loss, ctx.dev, ctx.scaler)
        return (grad0, grad1) + (None,) * 20


def pso_pair_loss(noise_pred_0, noise_pred_1, noise_ref_pred_0, noise_ref_pred_1, sample_0, sample_1, next_0, next_1,
                  timesteps_0, timesteps_1, human_prefer, *, scheduler=None, kind="turbo", beta=50.0, eps=0.1,
                  step_ratio=None, coefficients=None, loss_scale=1.0, return_stats=False, tune=(0, 0), grad_scaler=None):
    """Online PSO loss of one micro-step, differentiable w.r.t. ``noise_pred_0/1`` only.

    kind="turbo": ``scheduler.timesteps/.sigmas`` are read (EulerAncestral; T:810-837);
    kind="dmd":   ``scheduler.alphas_cumprod`` and ``prev_timestep = t - step_ratio`` (D:812-843);
    kind="affine": ``coefficients=((k0,a0,s0),(k1,a1,s1))`` per-sample float tensors.
    ``human_prefer`` is the [B,2] sign tensor of ``sample_compare`` / ``compare``.
    ``loss_scale`` folds accelerate's ``loss / gradient_accumulation_steps`` (T:857) into the
    same launch.  Returns ``loss`` (0-dim fp32) or ``(loss, stats[B,8])`` with
    stats = (logp_pol0, logp_ref0, logp_pol1, logp_ref1, delta0, delta1, z, pair_loss).
    ``grad_scaler`` (an ``amp.DeviceGradScaler``, fp16 training): the kernel computes the gradient already multiplied by
    the device scale S, so it is rounded to the prediction dtype scaled; the backward divides autograd's upstream factor
    by S, so ``grad_scaler.scale(loss).backward()`` leaves S x the gradient and ``loss.backward()`` the unscaled one.
    ``loss`` and ``stats`` are unscaled either way.
    """
    dev = _lib.require_cuda(noise_pred_0)
    ts0 = ts1 = tsp0 = tsp1 = c0 = c1 = None
    if kind == "affine":
        sched = runtime.affine_schedule(dev)
        c0, c1 = (torch.stack([v.to(device=dev, dtype=torch.float32).reshape(-1) for v in c]).contiguous()
                  for c in coefficients)
    else:
        ts0 = runtime.timesteps_on(timesteps_0, dev)
        ts1 = runtime.timesteps_on(timesteps_1, dev).to(ts0.dtype)
        if kind == "turbo":
            sched = runtime.turbo_schedule(scheduler, dev, _lib.ts_dtype_code(ts0))
        elif kind == "dmd":
            if step_ratio is None:
                raise ValueError("kind='dmd' needs step_ratio (train_online_pso_sdxl_dmd2.py:542)")
            sched = runtime.dmd_schedule(scheduler, dev, _lib.ts_dtype_code(ts0))
            tsp0, tsp1 = ts0 - step_ratio, ts1 - step_ratio  # D:816
        else:
            raise ValueError(f"unknown kind {kind!r}")
        B = noise_pred_0.shape[0]
        if ts0.numel() != B or ts1.numel() != B:
            raise _lib.Psob200Error(f"need one timestep per pair ({B}), got {ts0.numel()} / {ts1.numel()}")
    loss, stats = _OnlinePsoLoss.apply(noise_pred_0, noise_pred_1, noise_ref_pred_0.detach(), noise_ref_pred_1.detach(),
                                       sample_0.detach(), sample_1.detach(), next_0.detach(), next_1.detach(),
                                       ts0, ts1, tsp0, tsp1, c0, c1, human_prefer, sched, beta, eps, loss_scale,
                                       return_stats, tune, grad_scaler)
    return (loss, stats) if return_stats else loss


# ----------------------------------------------------------------------------- DreamBooth PSO
def edm_sigmas(noise_scheduler, timesteps: torch.Tensor, n_dim: int = 4, dtype=torch.float32) -> torch.Tensor:
    """``get_sigmas`` of the DreamBooth trainer (train_pso_sdxl_turbo_dreambooth.py:1675-1685): ``sigmas[i]`` for the schedule
    position ``i`` whose ``scheduler.timesteps[i] == t``, shaped ``[B, 1, 1, 1]``.  The reference finds ``i`` with one
    ``.nonzero().item()`` host sync per sample; here the lookup is one comparison matrix + argmax on the device, no sync
    (a timestep that is not in the schedule selects position 0 instead of raising)."""
    dev = timesteps.device
    sched_ts = noise_scheduler.timesteps.to(dev)
    sig = noise_scheduler.sigmas.to(device=dev, dtype=dtype)
    idx = (sched_ts[None, :] == timesteps.to(sched_ts.dtype)[:, None]).to(torch.uint8).argmax(dim=1)
    out = sig[idx].flatten()
    while out.dim() < n_dim:
        out = out.unsqueeze(-1)
    return out


class _DreamboothPsoLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, model_pred, ref_pred, noisy, target, sigmas, loss_type, beta_pso, neg_defactor,
                prior_loss_weight, loss_scale, tune, scaler):
        dev = _lib.require_cuda(model_pred, ref_pred, noisy, target, sigmas)
        b2, n = model_pred.shape[0], _n(model_pred)
        if b2 % 2:
            raise _lib.Psob200Error("DreamBooth-PSO batches are [win rows ; lose rows]: need an even row count")
        b = b2 // 2
        a = _lib.DreamboothArgs()
        mp = model_pred.contiguous()
        nz = noisy.contiguous()
        tg = target.contiguous() if target.dtype == nz.dtype else target.to(nz.dtype).contiguous()
        rp = None
        if loss_type == _lib.DB_PSO:
            rp = ref_pred.contiguous() if ref_pred.dtype == mp.dtype else ref_pred.to(mp.dtype).contiguous()
            a.ref_pred = rp.data_ptr()
        sg = sigmas.detach().to(device=dev, dtype=torch.float32).reshape(-1).contiguous()
        if sg.numel() != b2:
            raise _lib.Psob200Error(f"sigmas must have {b2} entries, got {sg.numel()}")
        grad = torch.empty(mp.shape, dtype=mp.dtype, device=dev)
        loss = torch.empty((), dtype=torch.float32, device=dev)
        stats = torch.empty((b, 8), dtype=torch.float32, device=dev)
        ws = runtime.workspace(dev, _lib.lib().psob200_pair_loss_workspace_bytes(b))
        a.model_pred, a.noisy, a.target, a.sigmas = mp.data_ptr(), nz.data_ptr(), tg.data_ptr(), sg.data_ptr()
        a.grad, a.loss, a.stats = grad.data_ptr(), loss.data_ptr(), stats.data_ptr()
        a.status = runtime.status_word(dev).data_ptr()
        a.workspace, a.workspace_bytes = ws.data_ptr(), ws.numel()
        a.b, a.N = b, n
        a.pred_dtype, a.latent_dtype, a.loss_type = _lib.dtype_code(mp), _lib.dtype_code(nz), loss_type
        a.beta_pso, a.neg_defactor = float(beta_pso), float(neg_defactor)
        a.prior_loss_weight, a.loss_scale = float(prior_loss_weight), float(loss_scale)
        a.tune_threads, a.tune_cluster = tune
        _launch_loss(dev, "psob200_dreambooth_pso_loss_grad", scaler, C.byref(a))
        del rp, tg, sg
        ctx.save_for_backward(grad)
        ctx.dev = dev
        ctx.scaler = scaler
        ctx.used = False
        ctx.mark_non_differentiable(stats)
        return loss, stats

    @staticmethod
    def backward(ctx, grad_loss, _grad_stats):
        if ctx.used:
            raise RuntimeError("pso_db_loss: backward may run only once (its gradient buffer is consumed)")
        ctx.used = True
        (grad,) = ctx.saved_tensors
        _apply_upstream((grad,), grad_loss, ctx.dev, ctx.scaler)
        return (grad,) + (None,) * 11


def pso_db_loss(model_pred, ref_pred, noisy_model_input, model_input, sigmas, *, loss_type="pso", beta_pso=1.0,
                neg_defactor=0.1, prior_loss_weight=0.0, loss_scale=1.0, tune=(0, 0), grad_scaler=None):
    """DreamBooth-PSO loss (train_pso_sdxl_turbo_dreambooth.py:1847-1865,1881-1935) on RAW UNet
    outputs: the EDM-style epsilon preconditioning ``x0_hat = -sigma*pred + noisy`` (:1855), the
    ``sigma^-2`` weighting (:1865), the win/lose chunking (:1891), the optional reference branch
    and the prior term all run in one kernel.  Rows [0,b) are win images, [b,2b) lose images.

    Returns ``(loss, model_losses_w[b], model_losses_l[b], logits[b])`` -- the three extras feed the
    logging at :1941-1950 and carry no gradient.  ``loss_type`` is "pso" or "pso_db"; anything else
    raises ValueError like :1929.  ``grad_scaler``: as in ``pso_pair_loss`` (fp16 loss scaling, :1953 under GradScaler).
    """
    if loss_type == "pso":
        lt = _lib.DB_PSO
        if ref_pred is None:
            raise ValueError("loss_type='pso' needs ref_pred (the adapter-disabled UNet output, :1897-1906)")
    elif loss_type == "pso_db":
        lt = _lib.DB_PSO_DB
    else:
        raise ValueError(f"Unknown loss type {loss_type}")
    loss, stats = _DreamboothPsoLoss.apply(model_pred, None if ref_pred is None else ref_pred.detach(),
                                           noisy_model_input.detach(), model_input.detach(), sigmas, lt, beta_pso,
                                           neg_defactor, prior_loss_weight, loss_scale, tune, grad_scaler)
    return loss, stats[:, 0], stats[:, 1], stats[:, 4]

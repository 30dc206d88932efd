"""Generates tests/golden/oracle_pins.npz: outputs of the oracle restatement on the inputs of the checks that once ran the
reference's own code next to it (TEST INFRASTRUCTURE).

    python -m oracle.make_golden_pins

Needs the reference (``oracle.reference_loader``): before anything is written, the restatement's outputs are checked against
the reference's code executed verbatim on the same inputs -- the sampler denoising loops and the DreamBooth micro-step
identical, the half-precision quirk of the distilled step within 1e-2 -- so that a changed oracle cannot be re-recorded
unnoticed.  The stored outputs keep that comparison with every later change of the oracle, on any machine without the
reference.  Each ``*_case`` function below is also what ``tests/test_oracle_golden.py`` runs, so inputs and outputs cannot
drift apart.
"""
from __future__ import annotations

import os

import numpy as np
import torch

from . import losses, reference_loader as rl, samplers, schedules, steps

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def bf16_quirk_case(reference_step=None):
    """The distilled step scored on bf16 latents without the upcast (the reference's behaviour on half inputs); with
    ``reference_step``, that function scores them instead of the restatement."""
    g = torch.Generator().manual_seed(123)
    x = torch.randn(2, 4, 8, 8, generator=g) * 3
    e = torch.randn(2, 4, 8, 8, generator=g)
    dsched = schedules.dmd_scheduler()
    td = torch.tensor([499, 249])
    xn, _ = steps.distilled_step(dsched, e, td, td - 250, x, generator=torch.Generator().manual_seed(9))
    if reference_step is None:
        _, lp = steps.distilled_step(dsched, e, td, td - 250, x.bfloat16(), prev_sample=xn.bfloat16(), upcast=False)
    else:
        _, lp = reference_step(dsched, e, td, td - 250, x.bfloat16(), prev_sample=xn.bfloat16(), device="cpu")
    return {"bf16_quirk_log_prob": lp.float()}


def _sampler_inputs():
    """A small fixed stand-in UNet and the initial latents of both sampler cases."""
    W = torch.randn(4, 4, generator=torch.Generator().manual_seed(3)) * 0.3
    unet = lambda x, t: torch.einsum("oc,bchw->bohw", W, x) * 0.5 + 0.1 * torch.tanh(x)
    return unet, torch.randn(2, 4, 8, 8, generator=torch.Generator().manual_seed(1))


def sampler_cases():
    """Both few-step sampler loops around a small fixed stand-in UNet, noise from seeded generators (turbo: one draw per
    sample; dmd: one draw shared by the batch)."""
    unet, lat0 = _sampler_inputs()
    B, shape = lat0.shape[0], tuple(lat0.shape[1:])
    g = torch.Generator().manual_seed(7)
    final, lats, lps, inputs = samplers.turbo_sampler(unet, schedules.turbo_scheduler(4), lat0,
                                                      [torch.randn(B, *shape, generator=g) for _ in range(4)], 4)
    out = {"turbo_final": final, "turbo_latents": torch.stack(lats), "turbo_log_probs": torch.stack(lps),
           "turbo_model_inputs": torch.stack(inputs)}
    ts, _ = schedules.dmd_distill_timesteps(4)
    g = torch.Generator().manual_seed(9)
    x0, lats, lps = samplers.dmd_sampler(unet, schedules.dmd_scheduler(), ts, lat0,
                                         [torch.randn(1, *shape, generator=g) for _ in range(3)])
    out.update({"dmd_x0": x0, "dmd_latents": torch.stack(lats), "dmd_log_probs": torch.stack(lps)})
    return out


def dreambooth_micro_step_case(loss_type, loss_fn=None):
    """BASELINE config 4's oracle micro-step (fixtures.micro_step.oracle_dreambooth_micro_step: tiny SDXL-architecture UNet,
    LoRA rank 4, b = 4, 2b rows) with the restated loss lines, or ``loss_fn``.  Returns (batch, outputs)."""
    from fixtures import micro_step, sdxl_unet
    from . import lora as olora
    torch.manual_seed(0)
    cfg = sdxl_unet.tiny_config()
    unet = sdxl_unet.UNet2DConditionModel(cfg)
    wrapped = olora.oracle_add_adapter(unet, 4, 4)
    g = torch.Generator().manual_seed(1)
    for m in wrapped:
        with torch.no_grad():
            m.lora_B["default"].weight.copy_(torch.randn(m.lora_B["default"].weight.shape, generator=g) * 0.03)
    unet.train()
    batch = micro_step.synth_dreambooth_batch(4, 32, cfg.cross_attention_dim, 32, 7, schedules.dreambooth_scheduler())
    loss, (lw, ll, logits) = micro_step.oracle_dreambooth_micro_step(olora, losses, unet, batch, loss_type=loss_type, beta_pso=5.0,
                                                                     neg_defactor=0.1, prior_loss_weight=0.5, loss_fn=loss_fn)
    grads = torch.cat([torch.cat([m.lora_A["default"].weight.grad.flatten(), m.lora_B["default"].weight.grad.flatten()])
                       for m in wrapped])
    sample = torch.randperm(grads.numel(), generator=torch.Generator().manual_seed(0))[:1024].sort().values  # keeps the file small
    p = f"dreambooth_{loss_type}_"
    return batch, {p + "loss": loss.detach(), p + "losses_w": lw.detach(), p + "losses_l": ll.detach(),
                   p + "logits": logits.detach(), p + "adapter_grad_norm": grads.norm(), p + "adapter_grad_sample": grads[sample]}


def check_against_reference(out):
    """``out`` (the restatement's outputs) against the reference's own code on the same inputs."""
    unet, lat0 = _sampler_inputs()
    sched = schedules.turbo_scheduler(4)
    ref = rl.pipeline_denoising_loop("turbo")(unet, sched, lat0 * sched.init_noise_sigma, torch.Generator().manual_seed(7), 4)
    assert torch.equal(out["turbo_final"], ref[0]) and torch.equal(out["turbo_latents"], torch.stack(ref[1]))
    assert torch.equal(out["turbo_model_inputs"], torch.stack(ref[3]))
    assert torch.allclose(out["turbo_log_probs"], torch.stack(ref[2]), rtol=1e-6)
    ts, _ = schedules.dmd_distill_timesteps(4)
    ref = rl.pipeline_denoising_loop("dmd")(unet, schedules.dmd_scheduler(), lat0.clone(), torch.Generator().manual_seed(9), 4,
                                          timesteps=ts)
    assert torch.equal(out["dmd_x0"], ref[0]) and torch.equal(out["dmd_latents"], torch.stack(ref[1]))
    assert torch.allclose(out["dmd_log_probs"], torch.stack(ref[2]), rtol=1e-6)
    lp_q = bf16_quirk_case(rl.distilled_step_with_logprob())["bf16_quirk_log_prob"]
    assert torch.allclose(lp_q, out["bf16_quirk_log_prob"], rtol=1e-2)
    for loss_type in ("pso", "pso_db"):
        got = dreambooth_micro_step_case(loss_type, rl.trainer_dreambooth_block())[1]
        assert all(torch.equal(got[k], out[k]) for k in got), loss_type


def main():
    if not rl.available():
        raise SystemExit("needs the reference (oracle.reference_loader): the recorded outputs are checked against it first")
    out = {}
    out.update(bf16_quirk_case())
    out.update(sampler_cases())
    for loss_type in ("pso", "pso_db"):
        out.update(dreambooth_micro_step_case(loss_type)[1])
    check_against_reference(out)
    path = os.path.join(OUT, "oracle_pins.npz")
    np.savez_compressed(path, **{k: v.numpy() for k, v in out.items()})
    print({k: tuple(v.shape) for k, v in out.items()}, os.path.getsize(path))


if __name__ == "__main__":
    main()

"""Load the reference's two step-with-logprob files verbatim (TEST INFRASTRUCTURE).

The files are executed from the read-only mount, never copied:

  /root/reference/human_preference_tuning/pso_pytorch/diffusers_patch/
      turbo_inference_with_logprob.py      (turbo_step_with_logprob, :24-116)
      distilled_inference_with_logprob.py  (distilled_step_with_logprob, :45-137)

Their only non-torch imports are ``randn_tensor`` and three scheduler class
names used purely as annotations (turbo :13-15, distilled :13-15); diffusers is
not installed in this image, so those names are provided by stub modules.

Only the fixture generators ``oracle/make_golden.py`` and ``oracle/make_golden_pins.py``
run this; ``available()`` says whether the reference is there.  The tests compare with the fixtures under
``tests/golden`` and need no copy of the reference.
"""
from __future__ import annotations

import importlib.util
import os
import sys
import types

import torch

REFERENCE_ROOT = os.environ.get("PSO_REFERENCE_ROOT", "/root/reference")
_PATCH_DIR = os.path.join(
    REFERENCE_ROOT, "human_preference_tuning", "pso_pytorch", "diffusers_patch"
)
_cache: dict[str, types.ModuleType] = {}


def available() -> bool:
    return os.path.isfile(os.path.join(_PATCH_DIR, "turbo_inference_with_logprob.py"))


def _randn_tensor(shape, generator=None, device=None, dtype=None, layout=None):
    # diffusers.utils.torch_utils.randn_tensor for a single generator on one device.
    return torch.randn(tuple(shape), generator=generator, device=device, dtype=dtype)


def _install_stub() -> None:
    if "diffusers" in sys.modules and not getattr(sys.modules["diffusers"], "_pso_oracle_stub", False):
        return  # a real diffusers is importable; use it
    names = {
        "diffusers": {"DDPMScheduler": type("DDPMScheduler", (), {})},
        "diffusers.utils": {},
        "diffusers.utils.torch_utils": {"randn_tensor": _randn_tensor},
        "diffusers.schedulers": {},
        "diffusers.schedulers.scheduling_euler_ancestral_discrete": {
            "EulerAncestralDiscreteScheduler": type("EulerAncestralDiscreteScheduler", (), {})
        },
        "diffusers.schedulers.scheduling_ddim": {
            "DDIMSchedulerOutput": type("DDIMSchedulerOutput", (), {}),
            "DDIMScheduler": type("DDIMScheduler", (), {}),
        },
    }
    for name, attrs in names.items():
        mod = types.ModuleType(name)
        mod._pso_oracle_stub = True
        for k, v in attrs.items():
            setattr(mod, k, v)
        sys.modules[name] = mod
    for name in names:
        if "." in name:
            parent, child = name.rsplit(".", 1)
            setattr(sys.modules[parent], child, sys.modules[name])


def _load(stem: str) -> types.ModuleType:
    if stem in _cache:
        return _cache[stem]
    if not available():
        raise FileNotFoundError(f"reference not mounted at {REFERENCE_ROOT}")
    _install_stub()
    path = os.path.join(_PATCH_DIR, stem + ".py")
    spec = importlib.util.spec_from_file_location("_pso_reference_" + stem, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    _cache[stem] = mod
    return mod


def turbo_step_with_logprob():
    """The reference's own function object (turbo_inference_with_logprob.py:24)."""
    return _load("turbo_inference_with_logprob").turbo_step_with_logprob


def distilled_step_with_logprob():
    """The reference's own function object (distilled_inference_with_logprob.py:45)."""
    return _load("distilled_inference_with_logprob").distilled_step_with_logprob


def get_x0_from_noise():
    """distilled_inference_with_logprob.py:36-42."""
    return _load("distilled_inference_with_logprob")._get_x0_from_noise


# ---------------------------------------------------------------------------------------------------------------------
# The trainers themselves cannot be imported (they need diffusers / peft / accelerate / ml_collections at module level),
# but the code of the hot path inside them can still be EXECUTED VERBATIM: the lines are read from the read-only mount at
# run time, dedented and exec'd in a namespace that provides exactly the names they use.  Nothing is copied into the repo;
# the blocks are located by their own first / last statements, not by line numbers.
# ---------------------------------------------------------------------------------------------------------------------
_TRAINERS = {
    "turbo": ("train_online_pso_sdxl_turbo.py", "turbo_step_with_logprob", "sample_compare"),
    "dmd": ("train_online_pso_sdxl_dmd2.py", "distilled_step_with_logprob", "compare"),
}


def _trainer_lines(kind: str) -> list[str]:
    path = os.path.join(REFERENCE_ROOT, "human_preference_tuning", _TRAINERS[kind][0])
    with open(path) as f:
        return f.read().split("\n")


def _dedent(block: list[str]) -> str:
    import textwrap
    return textwrap.dedent("\n".join(block)) + "\n"


def trainer_compare_fn(kind: str):
    """The reference's own ``sample_compare`` (turbo trainer :401-416) / ``compare`` (dmd2 trainer :420-434): the nested
    ``def`` is cut out of the trainer's ``main()`` and executed as is."""
    name = _TRAINERS[kind][2]
    lines = _trainer_lines(kind)
    start = next(i for i, l in enumerate(lines) if l.strip().startswith(f"def {name}(a, b):"))
    indent = len(lines[start]) - len(lines[start].lstrip())
    end = start + 1
    while end < len(lines) and (not lines[end].strip() or len(lines[end]) - len(lines[end].lstrip()) > indent):
        end += 1
    ns = {"torch": torch}
    exec(compile(_dedent(lines[start:end]), f"<reference {_TRAINERS[kind][0]}:{start + 1}-{end}>", "exec"), ns)
    return ns[name]


def trainer_loss_block(kind: str):
    """The micro-step's loss code of the reference's trainer, verbatim: from the first ``_, total_prob_0 = <step>(`` call
    through the closing ``)).mean()`` of the inline loss (turbo trainer :810-850, dmd2 trainer :812-854) -- four
    step-with-logprob calls, the compare function, the clamped ratios and the log-sigmoid loss.

    Returns ``run(noise_scheduler, preds, ref_preds, sample_0, sample_1, j, beta, eps, step_ratio=None) -> (loss, human_prefer)``
    where ``sample_k`` are dicts with the trainer's keys (``timesteps``, ``latents``, ``next_latents``, ``rewards``;
    tensors of shape [B, T, ...])."""
    fname, step_name, cmp_name = _TRAINERS[kind]
    lines = _trainer_lines(kind)
    start = next(i for i, l in enumerate(lines) if l.strip().startswith(f"_, total_prob_0 = {step_name}("))
    loss_at = next(i for i in range(start, len(lines)) if lines[i].strip().startswith("loss = -torch.log(torch.sigmoid("))
    end = next(i for i in range(loss_at, len(lines)) if lines[i].strip().startswith(")).mean()")) + 1
    code = compile(_dedent(lines[start:end]), f"<reference {fname}:{start + 1}-{end}>", "exec")
    step_fn = turbo_step_with_logprob() if kind == "turbo" else distilled_step_with_logprob()
    cmp_fn = trainer_compare_fn(kind)

    def cpu_step(*args, **kwargs):  # the trainer relies on the default device=cuda; everything else is untouched
        kwargs.setdefault("device", "cpu")
        return step_fn(*args, **kwargs)

    def run(noise_scheduler, preds, ref_preds, sample_0, sample_1, j, beta, eps, step_ratio=None):
        ns = {"torch": torch, step_name: cpu_step, cmp_name: cmp_fn, "noise_scheduler": noise_scheduler,
              "noise_pred_0": preds[0], "noise_pred_1": preds[1], "noise_ref_pred_0": ref_preds[0],
              "noise_ref_pred_1": ref_preds[1], "sample_0": sample_0, "sample_1": sample_1, "j": j, "step_ratio": step_ratio,
              "config": types.SimpleNamespace(train=types.SimpleNamespace(beta=beta, eps=eps))}
        exec(code, ns)
        return ns["loss"], ns["human_prefer"]

    run.source_span = (fname, start + 1, end)
    return run


def trainer_dreambooth_block():
    """The DreamBooth trainer's loss code, verbatim (personalization/train_pso_sdxl_turbo_dreambooth.py, from
    ``weighting = None`` through ``loss = loss + args.prior_loss_weight * prior_loss``: :1846-1935 -- EDM output
    preconditioning, per-sample weighted MSE, win / lose split, the reference-model branch, the ``pso`` / ``pso_db`` losses
    and the prior term).  The UNet call of the reference branch is served by a stub that returns the given raw
    reference prediction; ``accelerator.unwrap_model(unet).disable_adapters()`` / ``enable_adapters()`` are no-ops.

    Returns ``run(model_pred, ref_pred, noisy_model_input, model_input, sigmas, loss_type, beta_pso, neg_defactor,
    prior_loss_weight) -> (loss, model_losses_w, model_losses_l, logits)`` (raw UNet outputs in, like the trainer)."""
    import torch.nn.functional as F
    path = os.path.join(REFERENCE_ROOT, "personalization", "train_pso_sdxl_turbo_dreambooth.py")
    with open(path) as f:
        lines = f.read().split("\n")
    start = next(i for i, l in enumerate(lines) if l.strip() == "weighting = None")
    end = next(i for i in range(start, len(lines)) if lines[i].strip() == "loss = loss + args.prior_loss_weight * prior_loss") + 1
    code = compile(_dedent(lines[start:end]), f"<reference train_pso_sdxl_turbo_dreambooth.py:{start + 1}-{end}>", "exec")

    def run(model_pred, ref_pred, noisy_model_input, model_input, sigmas, loss_type, beta_pso, neg_defactor, prior_loss_weight):
        adapters = types.SimpleNamespace(disable_adapters=lambda: None, enable_adapters=lambda: None, set_adapter=lambda *_: None)
        ns = {"torch": torch, "F": F,
              "args": types.SimpleNamespace(do_edm_style_training=True, neg_defactor=neg_defactor, loss_type=loss_type,
                                            beta_pso=beta_pso, prior_loss_weight=prior_loss_weight),
              "scheduler_type": "EulerDiscreteScheduler",
              "noise_scheduler": types.SimpleNamespace(config=types.SimpleNamespace(prediction_type="epsilon")),
              "model_pred": model_pred, "noisy_model_input": noisy_model_input, "model_input": model_input, "sigmas": sigmas,
              "noise": None, "timesteps": None, "inp_noisy_latents": None, "prompt_embeds_input": None,
              "unet_added_conditions": None, "unet": lambda *a, **k: (ref_pred,),
              "accelerator": types.SimpleNamespace(unwrap_model=lambda m: adapters)}
        exec(code, ns)
        return ns["loss"], ns["model_losses_w"], ns["model_losses_l"], ns["logits"]

    run.source_span = ("train_pso_sdxl_turbo_dreambooth.py", start + 1, end)
    return run


def pipeline_denoising_loop(kind: str):
    """The denoising loop of the reference's sampler pipeline, verbatim: sdxl_turbo_with_logprob.py from
    ``all_latents = [latents]`` to the line before ``## vae decode`` (:111-149) / sdxl_dmd_with_logprob.py likewise
    (:108-162, with the file's own ``_get_x0_from_noise``).  The pipeline files import diffusers' pipeline classes at module
    level, so the loop is cut out and executed with the names it uses: the reference's own step function, a caller-supplied
    ``unet(latent_input, t) -> noise_pred`` behind the pipeline's call signature, the scheduler, the generator.

    Returns ``run(unet, noise_scheduler, latents, generator, num_inference_steps, timesteps=None)`` ->
    turbo: ``(latents, all_latents, all_log_probs, all_model_input_latents)``; dmd: ``(x0_pred, all_latents, all_log_probs)``.
    ``latents`` is what the pipeline holds when the loop starts (already multiplied by ``init_noise_sigma``)."""
    fname = "sdxl_turbo_with_logprob.py" if kind == "turbo" else "sdxl_dmd_with_logprob.py"
    with open(os.path.join(_PATCH_DIR, fname)) as f:
        lines = f.read().split("\n")
    start = next(i for i, l in enumerate(lines) if l.strip() == "all_latents = [latents]")
    end = next(i for i in range(start, len(lines)) if lines[i].strip().startswith("## vae decode"))
    code = compile(_dedent(lines[start:end]), f"<reference {fname}:{start + 1}-{end}>", "exec")
    ns0 = {"torch": torch}
    if kind == "dmd":
        d0 = next(i for i, l in enumerate(lines) if l.startswith("def _get_x0_from_noise("))
        d1 = next(i for i in range(d0 + 1, len(lines)) if lines[i].startswith("def ") or lines[i].startswith("@"))
        exec(compile("\n".join(lines[d0:d1]) + "\n", f"<reference {fname}:{d0 + 1}-{d1}>", "exec"), ns0)
    step_fn = turbo_step_with_logprob() if kind == "turbo" else distilled_step_with_logprob()
    step_name = "turbo_step_with_logprob" if kind == "turbo" else "distilled_step_with_logprob"

    def run(unet, noise_scheduler, latents, generator, num_inference_steps, timesteps=None):
        def unet_call(x, t, *args, **kwargs):  # the pipeline's two call conventions: [0] of a tuple / .sample
            out = unet(x, t)
            return (out,) if kwargs.get("return_dict") is False else types.SimpleNamespace(sample=out)

        ns = dict(ns0)
        ns.update({step_name: step_fn, "unet": unet_call, "noise_scheduler": noise_scheduler, "latents": latents,
                   "timesteps": noise_scheduler.timesteps if timesteps is None else timesteps, "generator": generator,
                   "num_inference_steps": num_inference_steps, "batch_size": latents.shape[0],
                   "prompt_embeds": torch.zeros(1), "unet_added_conditions": None})
        exec(code, ns)
        if kind == "turbo":
            return ns["latents"], ns["all_latents"], ns["all_log_probs"], ns["all_model_input_latents"]
        return ns["x0_pred"], ns["all_latents"], ns["all_log_probs"]

    run.source_span = (fname, start + 1, end)
    return run

"""bench.py's b200 arm on the tiny fixture (debug run, seconds): the JSON line carries the keys of the bench contract, the step
runs from the captured graph, kernels of this library were launched inside the timed region, and `--dump-outputs` writes what
the last timed step computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_b200_arm_json_line_on_the_tiny_fixture(built_lib, tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--tiny", "--config", "turbo64", "--steps", "6", "--warmup", "3",
                          "--no-cpu-baseline", "--no-kernel-figures", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                "dtype", "data", "config", "gpu_launches", "clocks", "e2e", "roofline", "lora_skinny_launches", "peak_hbm_gb"):
        assert key in line, key
    assert line["metric"] == "pso_train_pairs_per_sec" and line["unit"] == "pairs/s" and line["n_gpus"] == 1
    assert line["steps"] == 6 and line["warmup"] >= 3 and line["value"] > 0 and line["scaling"] == "weak"
    assert line["gpu_launches"] > 6 * 100  # 96 LoRA projections, forward + backward, every step
    e2e = line["e2e"]
    assert e2e["value"] > 0 and e2e["h2d_bytes_per_step"] > 0 and e2e["d2h_bytes_per_step"] == 4
    for r in (line["roofline"], line["lora_skinny_launches"]):
        assert r["bound"] in ("tensor", "hbm") and r["achieved"] > 0 and r["peak"] > 0
        assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-3 and r["launches_per_step"] > 0
    assert "workload" in line["config"] and line["clocks"]["sm_max_mhz"]
    # round 2: the backward of the timed step is not vacuous, and the reference's flow on the same GPU is reported next to it
    assert line["grad_norm"] > 0 and 0 < line["gate"]["open_fraction"] <= 1
    eager = line["gpu_eager_baseline"]
    assert eager["value"] > 0 and eager["ratio_ours_over_eager"] > 0
    par = eager["same_weights_parity"]  # both arms on the same adapters and batch (tiny fixture: bf16 noise of ~40 layers)
    assert par["loss_rel_diff"] <= 5e-2 and par["grad_cosine"] >= 0.9, par
    # --dump-outputs: the last timed step's loss and optimizer boundary (6 steps = one accumulation window), float arrays only
    dumped = {f[:-4]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert set(dumped) == {"loss", "grad_norm", "lora_params", "lora_grad", "adamw_exp_avg", "adamw_exp_avg_sq"}
    assert all(v.dtype in (np.float32, np.float64) for v in dumped.values())
    assert sum(v.nbytes for v in dumped.values()) <= 64 << 20
    assert abs(float(dumped["loss"]) * 6 - line["loss"]) <= 1e-5 * abs(line["loss"]) + 1e-6
    assert abs(float(dumped["grad_norm"][0]) - line["grad_norm"]) <= 1e-6 * line["grad_norm"]
    assert np.abs(dumped["adamw_exp_avg"]).max() > 0 and np.isfinite(dumped["lora_params"]).all()



def test_b200_arm_outputs_are_the_same_every_run(built_lib, tmp_path):
    """Same arguments, same outputs: two runs dump identical arrays (4 timed steps, no optimizer boundary among them, so the
    adapter gradient the steps accumulated is compared as well)."""
    for run in ("a", "b"):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--tiny", "--config", "turbo64", "--steps", "4",
                              "--warmup", "3", "--no-cpu-baseline", "--no-kernel-figures", "--no-eager-baseline",
                              "--dump-outputs", str(tmp_path / run)], capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-3000:]
    assert np.abs(np.load(tmp_path / "a" / "lora_grad.npy")).max() > 0
    for f in sorted(os.listdir(tmp_path / "a")):
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)), f

def test_b200_arm_dreambooth_config_on_the_tiny_fixture(built_lib):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--tiny", "--config", "dreambooth64", "--steps", "4", "--warmup", "3",
                          "--no-cpu-baseline", "--no-kernel-figures"], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["config"]["name"] == "dreambooth64" and line["config"]["loss_type"] == "pso" and line["value"] > 0
    assert line["grad_norm"] > 0 and line["gpu_launches"] > 0 and line["gpu_eager_baseline"]["value"] > 0
    assert line["gpu_eager_baseline"]["same_weights_parity"]["grad_cosine"] >= 0.9

"""bench.py's reference arm (CPU oracle port) on the tiny fixture: the JSON line carries every key the bench contract
names.  (The b200 arm needs a GPU; its line is checked on the box by the driver.)"""
import json
import os
import subprocess
import sys
import types

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line_has_the_contract_keys():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--tiny", "--config", "turbo64",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["metric"] == "pso_train_pairs_per_sec" and line["unit"] == "pairs/s"
    assert line["value"] > 0 and line["higher_is_better"] is True and line["vs_baseline"] is None
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1 and "workload" in line["config"]


def test_non_zero_ranks_of_the_reference_arm_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--tiny"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_dump_outputs_samples_long_buffers_at_fixed_positions(tmp_path, monkeypatch):
    """--dump-outputs on buffers longer than DUMP_SAMPLE (the SDXL case): the same seeded positions of every flat buffer, in
    ascending order, the same on every call; loss and gradient norm as they are."""
    sys.path.insert(0, ROOT)
    import bench
    monkeypatch.setattr(bench, "DUMP_SAMPLE", 64)
    n = 1000
    flat = torch.arange(n, dtype=torch.float32)
    opt = types.SimpleNamespace(flat_param=flat, exp_avg=2 * flat, exp_avg_sq=3 * flat, grad_norm=torch.tensor([0.5]))
    arm = types.SimpleNamespace(opt=opt, bucket=types.SimpleNamespace(flat=-flat), last_loss=torch.tensor(1.25),
                                dev=torch.device("cpu"))
    for run in ("a", "b"):
        bench.B200Arm.dump_outputs(arm, str(tmp_path / run))
    got = {f[:-4]: np.load(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")}
    assert set(got) == {"loss", "grad_norm", "lora_params", "lora_grad", "adamw_exp_avg", "adamw_exp_avg_sq"}
    assert all(v.dtype == np.float32 for v in got.values())
    assert float(got["loss"]) == 1.25 and got["grad_norm"].tolist() == [0.5]
    pos = got["lora_params"]  # the buffer holds its own index: the dump lists the sampled positions
    assert pos.shape == (64,) and np.all(np.diff(pos) >= 0) and pos.min() >= 0 and pos.max() < n and len(np.unique(pos)) > 32
    np.testing.assert_array_equal(got["lora_grad"], -pos)
    np.testing.assert_array_equal(got["adamw_exp_avg"], 2 * pos)
    np.testing.assert_array_equal(got["adamw_exp_avg_sq"], 3 * pos)
    for f in got:
        np.testing.assert_array_equal(got[f], np.load(tmp_path / "b" / (f + ".npy")))

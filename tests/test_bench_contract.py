"""bench.py prints exactly ONE JSON line on stdout with the contract keys: the CPU (reference) arm runs anywhere, the
CUDA arm on a GPU box."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
        "dtype", "data", "config", "cpu_baseline", "e2e"}


def run_bench(*args):
    r = subprocess.run([sys.executable, os.path.join(REPO, "bench.py"), *args], capture_output=True, text=True, cwd=REPO, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    return json.loads(lines[0])


def test_reference_arm_line():
    d = run_bench("--impl", "reference", "--steps", "1", "--warmup", "1")
    assert BASE <= set(d) and d["impl"] == "reference" and d["unit"] == "env-steps/s" and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["gpu_launches"] == 0


def test_dump_outputs_above_the_cap_is_a_fixed_sample_of_envs(tmp_path):
    import types

    import torch
    import bench
    n, cap = 1000, 4096 + 100 * (4 * 21 + 8)          # room for the .npy headers + 100 rows of 18 obs, rew, reset, time-out, id
    env = types.SimpleNamespace(num_envs=n, device="cpu", _global_env_offset=5000,
                                _obs_clamped=torch.arange(n * 18, dtype=torch.float32).reshape(n, 18),
                                rew_buf=torch.arange(n, dtype=torch.float32), reset_buf=torch.arange(n) % 2,
                                timeout_buf=torch.arange(n) % 3 == 0)
    for d in ("a", "b"):
        bench.dump_outputs(env, str(tmp_path / d), max_bytes=cap)
    names = ("obs", "rew", "reset", "time_outs", "env_ids")
    a, b = ({k: np.load(tmp_path / d / f"{k}.npy") for k in names} for d in ("a", "b"))
    assert all(np.array_equal(a[k], b[k]) for k in names) and sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= cap
    rows = a["rew"].astype(np.int64)
    assert len(rows) == 100 and np.all(np.diff(rows) > 0) and np.array_equal(a["env_ids"], rows + 5000)
    assert np.array_equal(a["obs"], env._obs_clamped.numpy()[rows]) and np.array_equal(a["reset"], rows % 2)
    assert np.array_equal(a["time_outs"], rows % 3 == 0) and all(v.dtype in (np.float32, np.float64) for v in a.values())


@pytest.mark.gpu
def test_cuda_arm_line(tmp_path):
    d = run_bench("--steps", "5", "--warmup", "3", "--no-sweep", "--ppo-iters", "3", "--num-envs", "65536", "--e2e-steps", "3",
                  "--dump-outputs", str(tmp_path))
    # the outputs of the last timed step, every env (65,536 x 84 B is under the 64 MB cap, so no sampling)
    out = {k: np.load(tmp_path / f"{k}.npy") for k in ("obs", "rew", "reset", "time_outs", "env_ids")}
    assert out["obs"].shape == (65536, 18) and all(out[k].shape == (65536,) for k in ("rew", "reset", "time_outs", "env_ids"))
    assert all(a.dtype in (np.float32, np.float64) and np.isfinite(a).all() for a in out.values())
    assert np.array_equal(out["env_ids"], np.arange(65536)) and np.abs(out["obs"]).max() <= 5.0 and out["obs"].std() > 0
    assert set(np.unique(out["reset"])) <= {0.0, 1.0} and set(np.unique(out["time_outs"])) <= {0.0, 1.0}
    assert BASE | {"roofline", "clocks", "gpu_launches", "ppo", "ppo_frames_per_s"} <= set(d)
    assert d["n_gpus"] == 1 and d["steps"] == 5 and d["warmup"] >= 3 and d["gpu_launches"] == 5 and d["scaling"] == "weak"
    assert d["value"] > 1e8 and d["e2e"]["value"] > 1e7 and d["e2e"]["h2d_bytes_per_step"] == 65536 * 8
    r = d["roofline"]          # the BINDING resource of the env step (FP32, SURVEY §8d); HBM rides along as roofline_hbm
    assert r["bound"] == "fp32_fma" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and r["unit"] == "TFLOP/s"
    assert 0.1 < r["frac"] < 1.0 and r["flops_per_env_step"] > 1e4
    h = d["roofline_hbm"]
    assert h["bound"] == "hbm" and h["unit"] == "GB/s" and abs(h["frac"] - h["achieved"] / h["peak"]) < 1e-9
    c1 = d["cpu_baseline_c1"]  # reference's unmodified Python step, configs[0] (committed build-container record on the GPU box)
    assert c1 and c1["value"] > 0 and "64 envs x 200 control steps" in c1["sample"] and c1["measured_on"]
    u = d["ppo"]["reference_network"]["update_roofline"]
    assert u["bound"] == "tensor" and abs(u["frac"] - u["achieved"] / u["peak"]) < 1e-9
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] > 0
    assert "hw_slowdown" not in d["clocks"]["reasons"]
    p = d["ppo"]["reference_network"]
    assert p["value"] == d["ppo_frames_per_s"] > 1e6 and p["network"].startswith("mlp[256,128,64]+lstm256") and p["cuda_graphs"]
    assert "hand-written" in p["update"]

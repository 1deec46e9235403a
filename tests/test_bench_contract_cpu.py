"""bench.py's reference arm (the CPU oracle port on the host cores) runs without a GPU and prints ONE JSON line carrying the
keys the driver reads; without a GPU the product arm refuses instead of falling back to the CPU."""
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "env-steps/s" and d["higher_is_better"] is True and d["value"] > 0
    assert d["metric"] == "stage03 env-steps/sec" and "exp02_v2_full" in d["config"]["workload"]
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["steps"] == 1 and d["warmup"] == 0 and d["n_gpus"] == 1 and d["vs_baseline"] is None


def test_steps_and_dump_outputs_arguments_are_checked(tmp_path):
    for args in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path)]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=120, cwd=ROOT)
        assert out.returncode == 2 and not out.stdout.strip(), (args, out.stderr[-2000:])
    assert not os.listdir(tmp_path)


def test_dump_outputs_writes_a_seeded_sample_in_float32_or_float64(tmp_path, monkeypatch):
    import numpy as np
    import bench
    E = 1000
    arrays = {"obs_lidar": torch.rand(E, 3, 13, 26), "reward": torch.rand(E), "done": torch.arange(E, dtype=torch.uint8) % 2,
              "info": torch.arange(E * 8, dtype=torch.int32).reshape(E, 8)}
    bench.dump_outputs(str(tmp_path / "all"), arrays, seed=5)
    got = {f[:-4]: np.load(tmp_path / "all" / f) for f in os.listdir(tmp_path / "all")}
    assert sorted(got) == ["done", "env_index", "info", "obs_lidar", "reward"]
    assert got["obs_lidar"].dtype == np.float32 and got["info"].dtype == np.float64 and got["done"].dtype == np.float64
    assert np.array_equal(got["env_index"], np.arange(E)) and np.array_equal(got["info"], arrays["info"].numpy())
    monkeypatch.setattr(bench, "DUMP_BUDGET_BYTES", 100 * (3 * 13 * 26 * 4 + 4 + 8 + 64 + 8))      # room for 100 envs
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), arrays, seed=5)
    a = {f[:-4]: np.load(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")}
    b = {f[:-4]: np.load(tmp_path / "b" / f) for f in os.listdir(tmp_path / "b")}
    rows = a["env_index"].astype(np.int64)
    assert len(rows) == 100 and np.all(np.diff(rows) > 0) and all(np.array_equal(a[k], b[k]) for k in a)
    assert np.array_equal(a["obs_lidar"], arrays["obs_lidar"].numpy()[rows]) and np.array_equal(a["reward"], arrays["reward"].numpy()[rows])


def test_product_arm_refuses_without_a_gpu():
    if torch.cuda.is_available():
        import pytest
        pytest.skip("GPU present")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode != 0 and "no CPU fallback" in (out.stderr + out.stdout)
    assert not [l for l in out.stdout.splitlines() if l.strip().startswith("{")]      # no number is printed

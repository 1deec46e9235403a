"""bench.py on the GPU: --steps sets the timed steps, and --dump-outputs writes the same outputs on every run with the same
arguments, so that two builds can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(*args):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    return json.loads(lines[0])


@pytest.mark.parametrize("preset,lidar_key", [("exp02_v2_full", "obs_lidar"), ("level5_c1", "obs_stacked_spheres")])
def test_dump_outputs_repeat_run_to_run(tmp_path, preset, lidar_key):
    args = ["--preset", preset, "--envs", "2048", "--steps", "7", "--warmup", "3", "--spinup", "20",
            "--no-cpu", "--no-e2e", "--no-also", "--no-rollout"]
    runs = []
    for name in ("a", "b"):
        line = _bench(*args, "--dump-outputs", str(tmp_path / name))
        assert line["steps"] == 7 and line["gpu_launches"] >= 7
        runs.append({f[:-4]: np.load(tmp_path / name / f) for f in sorted(os.listdir(tmp_path / name))})
    a, b = runs
    assert {lidar_key, "obs_inertial_data", "obs_last_action", "reward", "done", "info", "env_index"} <= set(a)
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    n = len(a["env_index"])
    assert all(v.shape[0] == n for v in a.values()) and a["obs_inertial_data"].shape == (n, 15)
    assert a.keys() == b.keys() and all(np.array_equal(a[k], b[k]) for k in a)

"""Cost of the ray-cast LiDAR as the agent's sensor: one env step (dc_step, auto-reset, random actions) in the fused flavour
and with lidar="raycast", timed on one GPU with CUDA events after warm-up, median of --repeats windows.  The two envs live
side by side and their windows alternate inside each repeat, so both see the same machine state.

Workloads: exp02_v2_full at 65,536 envs (radii 0.1 m for wingmen and munitions) and swarm (4 wingmen, 64 munitions) at
8,192 envs (same radii).  The ray-cast step also runs raycast_sphere_kernel, which rewrites every updated env's whole
sphere: 3 x 338 floats = 4,056 B per env (lidar_ids is not bound here), an estimate of its stores, not a measurement.
The card name and nvidia-smi's power limit / max SM clock are read in the same run and written beside the numbers.

    python profiles/raycast_env_bench.py --out profiles/raycast_env_b200.json
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

WORKLOADS = (("exp02_v2_full", 65536), ("swarm", 8192))


def _median(xs):
    xs = sorted(xs)
    return xs[len(xs) // 2]


def _window(env, actions, n):
    """ms per step over one window of n back-to-back steps."""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(n):
        env.step(actions[i % len(actions)])
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / n


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--repeats", type=int, default=7)
    p.add_argument("--steps", type=int, default=50, help="steps per timed window")
    p.add_argument("--warmup", type=int, default=30)
    p.add_argument("--radius", type=float, default=0.1)
    p.add_argument("--out", required=True)
    a = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("raycast_env_bench: needs a CUDA device (nothing here is measured on the CPU)")
    from dronechase_b200 import BatchedThreatEngageEnv, preset

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True)
    result = {"device": torch.cuda.get_device_name(0), "nvidia_smi": smi.stdout.strip(), "repeats": a.repeats,
              "steps_per_window": a.steps, "radius_m": a.radius, "workloads": []}
    for name, E in WORKLOADS:
        envs = {"fused": BatchedThreatEngageEnv(preset(name), n_envs=E, seed=1, device=0, auto_reset=True),
                "raycast": BatchedThreatEngageEnv(preset(name, lidar="raycast", ray_radius=(a.radius, a.radius)), n_envs=E, seed=1,
                                                  device=0, auto_reset=True)}
        g = torch.Generator(device="cuda"); g.manual_seed(0)
        actions = []
        for _ in range(16):
            x = torch.rand(E, 4, generator=g, device="cuda") * 2 - 1
            x[:, 3] = (x[:, 3] + 1) / 2
            actions.append(x)
        for env in envs.values():
            env.reset()
            _window(env, actions, a.warmup)
        times = {k: [] for k in envs}
        for _ in range(a.repeats):
            for k, env in envs.items():
                times[k].append(_window(env, actions, a.steps))
        marked = {k: float((env.obs["lidar"][:, 0] < 1).sum(dim=(1, 2)).float().mean()) for k, env in envs.items()}
        row = {"preset": name, "envs": E, "ms_per_step": {k: _median(v) for k, v in times.items()},
               "windows_ms": times, "marked_cells_per_env_last_step": marked}
        row["raycast_over_fused"] = row["ms_per_step"]["raycast"] / row["ms_per_step"]["fused"]
        row["added_ms"] = row["ms_per_step"]["raycast"] - row["ms_per_step"]["fused"]
        result["workloads"].append(row)
        print(json.dumps(row), flush=True)
        for env in envs.values():
            env.close()
    with open(a.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({k: v for k, v in result.items() if k != "workloads"}))


if __name__ == "__main__":
    main()

"""Policy-driven wingmen on the device, timed on one GPU with CUDA events after warm-up (median of --repeats windows).

Workload: the level4 evaluation task with two "nn" drivers (config.evaluation_preset, Evaluation_Task defaults otherwise) at
--envs envs, auto-reset, one LidarInertialActionPolicy per slot (reference defaults: 256 features, pi 128/256/512, Tanh;
different weights per slot).  Three ways to serve the two slots through drivers.TaskDrivers:

  module   the torch float32 module (torch's default backend flags: cuDNN convolutions may use TF32, matmuls do not)
  copies   FusedPolicy (dc_policy_forward) on contiguous copies of the slot's rows: what a caller had before serve existed
  serve    FusedPolicy handed to TaskDrivers directly: dc_policy_serve, one launch per slot, slabs read in place

For each: TaskDrivers.serve (dc_lw_observe + the two policy slots) and a full TaskDrivers.step (serve + dc_step + the
auto-reset zeroing of last_action); dc_lw_observe + dc_step alone are timed for reference.  The variants alternate inside
each repeat and share one env.  The fused variants run in "3xtf32" (float32-grade, the default) and again in "tf32".
The card name and nvidia-smi's power limit / max SM clock are read in the same run and written beside the numbers.

    python profiles/wingman_serve_bench.py --out profiles/wingman_serve_b200.json
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def _median(xs):
    xs = sorted(xs)
    return xs[len(xs) // 2]


def _window(fn, n):
    """ms per call over one window of n back-to-back calls."""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / n


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--envs", type=int, default=65536)
    p.add_argument("--repeats", type=int, default=7)
    p.add_argument("--calls", type=int, default=10, help="calls per timed window")
    p.add_argument("--out", required=True)
    a = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("wingman_serve_bench: needs a CUDA device (nothing here is measured on the CPU)")
    from dronechase_b200 import BatchedThreatEngageEnv
    from dronechase_b200.config import evaluation_preset
    from dronechase_b200.drivers import TaskDrivers
    from dronechase_b200.policy import LidarInertialActionPolicy

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True)
    configuration = {"drivers": [{"type": "nn", "name": "nn_1"}, {"type": "nn", "name": "nn_2"}]}
    res = {"device": torch.cuda.get_device_name(0), "nvidia_smi": smi.stdout.strip(), "envs": a.envs, "repeats": a.repeats,
           "calls_per_window": a.calls, "workload": "evaluation_preset, drivers nn + nn, auto_reset, default network per slot"}
    env = BatchedThreatEngageEnv(evaluation_preset(configuration), n_envs=a.envs, seed=1, device=0, auto_reset=True)
    env.reset()
    slots = env.cfg.policy_slots
    mods = {j: LidarInertialActionPolicy(env=env, seed=100 + j) for j in slots}

    def copies(f):
        return lambda obs: f({k: v.contiguous() for k, v in obs.items()})

    def observe_and_step():
        env.lw_observe()
        env.step(None)

    variants = {"module": TaskDrivers(env, mods)}
    for prec in ("3xtf32", "tf32"):
        fused = {j: m.fused(prec) for j, m in mods.items()}
        variants[f"copies_{prec}"] = TaskDrivers(env, {j: copies(f) for j, f in fused.items()})
        variants[f"serve_{prec}"] = TaskDrivers(env, fused)
    for drv in variants.values():                         # warm-up: every shape, cuDNN's algorithm choice
        for _ in range(3):
            drv.serve(); drv.step(None)
    for _ in range(3):
        observe_and_step()
    torch.cuda.synchronize()
    t_serve = {k: [] for k in variants}
    t_step = {k: [] for k in variants}
    t_env = []
    for _ in range(a.repeats):                            # alternating
        for k, drv in variants.items():
            t_serve[k].append(_window(drv.serve, a.calls))
            t_step[k].append(_window(lambda: drv.step(None), a.calls))
        t_env.append(_window(observe_and_step, a.calls))
    res["ms_per_call"] = {k: {"TaskDrivers.serve": _median(t_serve[k]), "TaskDrivers.step": _median(t_step[k])} for k in variants}
    res["ms_per_call"]["env_only"] = {"lw_observe + step": _median(t_env)}
    res["ms_all"] = {"serve": t_serve, "step": t_step, "env_only": t_env}
    m = res["ms_per_call"]
    res["speedup"] = {prec: {"serve_vs_module": m["module"]["TaskDrivers.serve"] / m[f"serve_{prec}"]["TaskDrivers.serve"],
                             "serve_vs_copies": m[f"copies_{prec}"]["TaskDrivers.serve"] / m[f"serve_{prec}"]["TaskDrivers.serve"],
                             "step_vs_module": m["module"]["TaskDrivers.step"] / m[f"serve_{prec}"]["TaskDrivers.step"],
                             "step_vs_copies": m[f"copies_{prec}"]["TaskDrivers.step"] / m[f"serve_{prec}"]["TaskDrivers.step"]}
                      for prec in ("3xtf32", "tf32")}
    res["note"] = ("per call, CUDA events around back-to-back calls; the two slots' slabs (65,536 x 2 x 4 KB spheres = 532 MB) "
                   "exceed the 126 MB L2; the env state evolves across windows (the variants share it, alternating)")
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "ms_all"}, indent=1))
    env.close()


if __name__ == "__main__":
    main()

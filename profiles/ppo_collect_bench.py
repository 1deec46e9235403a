"""PPO rollout collection on the device, timed on one GPU with CUDA events after warm-up (median of --repeats).

  1. dc_policy_forward (clipped mean action) vs dc_policy_act (sample = 1: action, log-prob, value), both precisions, at
     --envs envs, on LidarInertialActorCritic defaults (features 256, pi = vf = 128/256/512).  Shape arithmetic predicts
     about 1.46x for act: the value branch adds ~197 k MACs per env to ~425 k.
  2. PPORollout.collect vs DeviceRollout.collect(fused) on exp02_v2_full, T = 16, in env-steps/s (alternating).
  3. dc_gae at T = 128 vs the same recurrence as a torch loop, with the bytes it must move (17 B per (t, env)).

The card name and nvidia-smi's power limit / max SM clock are read in the same run and written beside the numbers.

    python profiles/ppo_collect_bench.py --out profiles/ppo_collect_b200.json
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


def _time(fn, n, repeats):
    """Median over `repeats` windows of n calls: ms per call."""
    out = []
    for _ in range(repeats):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        b.record()
        b.synchronize()
        out.append(a.elapsed_time(b) / n)
    return _median(out), out


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--envs", type=int, default=65536)
    p.add_argument("--repeats", type=int, default=7)
    p.add_argument("--preset", default="exp02_v2_full")
    p.add_argument("--out", required=True)
    a = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ppo_collect_bench: needs a CUDA device (nothing here is measured on the CPU)")
    from dronechase_b200 import BatchedThreatEngageEnv, _lib
    from dronechase_b200.policy import LidarInertialActorCritic
    from dronechase_b200.rollout import DeviceRollout, PPORollout
    from tests.test_gpu_policy import _obs

    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True)
    res = {"device": torch.cuda.get_device_name(0), "nvidia_smi": smi.stdout.strip(), "envs": a.envs, "repeats": a.repeats}
    E = a.envs

    # ---- 1. the kernels
    ac = LidarInertialActorCritic(seed=0, device="cuda")
    obs = _obs(E, 3, seed=1)
    f32 = dict(dtype=torch.float32, device="cuda")
    act_out = dict(env_actions=torch.empty(E, 4, **f32), raw_actions=torch.empty(E, 4, **f32), log_prob=torch.empty(E, **f32),
                   value=torch.empty(E, **f32))
    kern = {}
    for prec in ("3xtf32", "tf32"):
        fused = ac.fused(prec)
        out = torch.empty(E, 4, **f32)
        fwd = lambda: fused(obs, out=out)                                           # noqa: E731
        act = lambda: fused.act(obs, 0, seed=1, **act_out)                          # noqa: E731
        for _ in range(5):
            fwd(); act()
        t_f, t_a = [], []
        for _ in range(a.repeats):                                                  # alternating
            t_f.append(_time(fwd, 20, 1)[0]); t_a.append(_time(act, 20, 1)[0])
        kern[prec] = {"dc_policy_forward_ms": _median(t_f), "dc_policy_act_ms": _median(t_a), "ratio": _median(t_a) / _median(t_f),
                      "forward_ms_all": t_f, "act_ms_all": t_a}
        fused.close()
    res["kernels"] = kern
    res["kernels_note"] = ("per launch, CUDA events around 20 back-to-back launches; inputs 65,536 x 4 KB spheres = 268 MB, "
                           "more than the 126 MB L2")

    # ---- 2. collection
    env = BatchedThreatEngageEnv(a.preset, n_envs=E, seed=1234, device=0, auto_reset=True, with_hits=True)
    env.reset()
    T = 16
    ac_env = LidarInertialActorCritic(env=env, seed=1234)
    fused = ac_env.fused()
    plain, ppo = DeviceRollout(env, T), PPORollout(env, T, seed=1)
    plain.collect(fused, n_steps=4); ppo.collect(fused, n_steps=4)
    t_plain, t_ppo = [], []
    for _ in range(a.repeats):
        t_plain.append(_time(lambda: plain.collect(fused), 1, 1)[0]); t_ppo.append(_time(lambda: ppo.collect(fused), 1, 1)[0])
    res["collect"] = {"preset": a.preset, "steps": T, "unit": "env-steps/s",
                      "DeviceRollout.collect(fused)": E * T / (_median(t_plain) * 1e-3),
                      "PPORollout.collect(fused)": E * T / (_median(t_ppo) * 1e-3),
                      "ms_all": {"DeviceRollout": t_plain, "PPORollout": t_ppo},
                      "note": "PPORollout also computes V(s_T) after the loop (one more launch)"}
    fused.close(); env.close()
    del plain, ppo

    # ---- 3. GAE
    TG = 128
    g = torch.Generator(device="cuda").manual_seed(0)
    rewards = torch.randn(TG, E, generator=g, device="cuda")
    values = torch.randn(TG, E, generator=g, device="cuda")
    dones = (torch.rand(TG, E, generator=g, device="cuda") < 0.02).to(torch.uint8)
    last_values = torch.randn(E, generator=g, device="cuda")
    adv, ret = torch.empty_like(rewards), torch.empty_like(rewards)
    import ctypes as C
    L = _lib.lib()
    ptr = lambda t: C.c_void_p(t.data_ptr())                                       # noqa: E731
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def gae_cuda():
        _lib.check(L.dc_gae(ptr(rewards), ptr(dones), ptr(values), ptr(last_values), TG, E, 0.99, 0.95, ptr(adv), ptr(ret), stream), "dc_gae")

    adv_t = torch.empty_like(rewards)

    def gae_torch():
        a_ = torch.zeros(E, device="cuda")
        next_v = last_values
        nonterm = 1.0 - dones.float()
        for t in range(TG - 1, -1, -1):
            a_ = rewards[t] + 0.99 * next_v * nonterm[t] - values[t] + 0.99 * 0.95 * nonterm[t] * a_
            adv_t[t] = a_
            next_v = values[t]
        return adv_t + values

    for _ in range(3):
        gae_cuda(); gae_torch()
    t_c, _ = _time(gae_cuda, 20, a.repeats)
    t_t, _ = _time(gae_torch, 3, a.repeats)
    torch.cuda.synchronize()
    bytes_ = 17 * TG * E
    res["gae"] = {"T": TG, "E": E, "dc_gae_ms": t_c, "torch_loop_ms": t_t, "speedup": t_t / t_c, "bytes": bytes_,
                  "dc_gae_GBps": bytes_ / (t_c * 1e-3) / 1e9,
                  "hbm_share_of_7.7TBps": bytes_ / (t_c * 1e-3) / 7.7e12,
                  "max_abs_diff_vs_torch_loop": float((adv - adv_t).abs().max()),
                  "note": "17 B per (t, env): rewards, values, advantages, returns float32 + dones uint8; inputs 39 MB + outputs 67 MB "
                          "fit the 126 MB L2 after the first pass, so repeated calls may be served partly from L2"}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: v for k, v in res.items() if k != "collect"} | {"collect": {k: v for k, v in res["collect"].items() if k != "ms_all"}},
                     default=str)[:3000])


if __name__ == "__main__":
    main()

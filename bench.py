#!/usr/bin/env python
"""Benchmark of the stage03 env step: env-steps/s on N B200s, next to the CPU oracle.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--envs E_per_gpu] [--preset exp02_vFinal] [--dump-outputs DIR]
    python bench.py --impl reference ...      # the CPU arm on the box's host cores

One "step" = one pass of the hot path (Env.step of the reference, 16 physics substeps + logic +
observation) over every env of the shard.  N > 1 is launched by torchrun (one rank per GPU): envs are
sharded by index range with no collective on the step path; the only collective is one NCCL
all-reduce of the episode statistics after the timed region.  Rank 0 prints ONE JSON line.

--dump-outputs DIR writes what the last timed step returned (rank 0's shard) as DIR/<name>.npy, so that two builds can
be compared output for output: the same arguments give the same seeded actions, hence the same inputs, on every run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "stage03 env-steps/sec"
UNIT = "env-steps/s"


def algorithmic_bytes_per_env_step(n_lw: int, n_lm: int, lidar_channels: int) -> int:
    """DESIGN.md 'algorithmic bytes': per drone 11 state quads read + 11 written (16 B each), the
    formation quad for wingmen, 64 B env scalars in and out, action, observation, reward/done/info."""
    D = n_lw + n_lm
    state = D * 2 * 11 * 16 + n_lw * 2 * 16
    obs = lidar_channels * 13 * 26 * 4 + 15 * 4 + 4 * 4
    return state + 2 * 64 + 16 + obs + 4 + 1 + 32


def algorithmic_bytes_level5(n_lw: int, n_lm: int, multi_obs: int = 0, student: bool = False) -> int:
    """level5 adds to the level4 figure: the stacked observation (6,3,13,26) + mask written in full, this step's ring
    entries written (per wingman: 32 B pose + D x (4 B meta + 24 B feature)) and up to five entries read back.
    ``student``: a second stack + mask per step.  ``multi_obs`` 1 (Level5DumbMultiObs): one stack, mask, inertial vector and
    teacher action per wingman instead of the agent's, and five ring entries read back per observer; 2
    (Level52BTEvaluationEnvironment): no observation at all (the ring entries are still written)."""
    D = n_lw + n_lm
    entry = 32 + D * 28
    base = algorithmic_bytes_per_env_step(n_lw, n_lm, 0)
    stack = 6 * 3 * 13 * 26 * 4 + 6
    if multi_obs == 2:
        return base + n_lw * entry
    if multi_obs == 1:
        return base + n_lw * (stack + 60 + 16 + 1 + 5 * entry) + n_lw * entry
    return base + stack * (2 if student else 1) + n_lw * entry + 5 * entry * (2 if student else 1) + 2 * 32


class ClockSampler:
    """nvidia-smi clocks/throttle reasons while the timed region runs (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = sorted(int(r[1]) for r in self.rows if len(r) >= 8 and r[1].isdigit())
        mx = [int(r[2]) for r in self.rows if len(r) >= 8 and r[2].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) >= 8 for n, v in zip(names, r[4:8]) if v.lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": reasons}


DUMP_BUDGET_BYTES = 48 << 20          # what --dump-outputs writes in all stays under 64 MB


def dump_outputs(folder, arrays, seed=0):
    """Write ``arrays`` (name -> device tensor whose first axis is the env) as ``folder/<name>.npy``: float32 tensors as
    float32, every other dtype as float64 (exact for the bool / uint8 / int32 outputs).  When all envs would exceed
    DUMP_BUDGET_BYTES, the same fixed, seeded sample of env rows is taken from every array; ``env_index.npy`` lists the
    rows written."""
    import numpy as np
    import torch
    E = next(iter(arrays.values())).shape[0]
    per_env = sum((4 if t.dtype == torch.float32 else 8) * (t.numel() // E) for t in arrays.values()) + 8
    n = min(E, max(1, DUMP_BUDGET_BYTES // per_env))
    rows = np.arange(E) if n == E else np.sort(np.random.RandomState(seed).choice(E, n, replace=False))
    os.makedirs(folder, exist_ok=True)
    idx = torch.from_numpy(rows).to(next(iter(arrays.values())).device)
    for name, t in arrays.items():
        a = t.index_select(0, idx).cpu().numpy()
        np.save(os.path.join(folder, name + ".npy"), a if a.dtype == np.float32 else a.astype(np.float64))
    np.save(os.path.join(folder, "env_index.npy"), rows.astype(np.float64))


# --------------------------------------------------------------------------------------------- CPU arm
_W = {}


def _cpu_init(preset, n_envs, seed, counter):
    """Pool initialiser: every worker process owns one oracle batch for the whole run."""
    import dataclasses
    import numpy as np
    from oracle.env_oracle import EnvOracle, PRESETS
    with counter.get_lock():
        idx = counter.value
        counter.value += 1
    if preset.startswith("stage02"):
        from oracle.stage02_oracle import STAGE02, Stage02Oracle
        n_lm = 10 if preset.endswith("10lm") else 5
        orc = Stage02Oracle(dataclasses.replace(STAGE02, n_lm=n_lm, initial_round=n_lm), n_envs, seed=seed,
                            env_offset=idx * n_envs, auto_reset=True)
    elif preset.startswith("level5"):
        from oracle.level5_oracle import LEVEL5_C1, LEVEL5_DUMB, LEVEL5_EVAL2BT, LEVEL5_FUSION, Level5Oracle
        cfg5 = {"level5_fusion": LEVEL5_FUSION, "level5_dumb_multiobs": LEVEL5_DUMB, "level5_eval_2bt": LEVEL5_EVAL2BT}.get(preset, LEVEL5_C1)
        orc = Level5Oracle(cfg5, n_envs, seed=seed, env_offset=idx * n_envs, auto_reset=True)
    elif preset == "stage01":
        from oracle.stage01_oracle import Stage01Oracle
        orc = Stage01Oracle(n_envs=n_envs, seed=seed, env_offset=idx * n_envs, auto_reset=True)
    else:
        orc = EnvOracle(PRESETS[preset], n_envs, seed=seed, env_offset=idx * n_envs, auto_reset=True)
    orc.reset()
    _W.update(orc=orc, rng=np.random.RandomState(seed + idx), n=n_envs, np=np)


def _cpu_advance(inner):
    np, rng, n, orc = _W["np"], _W["rng"], _W["n"], _W["orc"]
    t0 = time.perf_counter()
    for _ in range(inner):
        a = np.concatenate([rng.uniform(-1, 1, (n, 3)), rng.uniform(0, 1, (n, 1))], axis=1)
        orc.step(a)
    return time.perf_counter() - t0


class CpuOracleArm:
    """The numpy float64 oracle (restated CPU port of the reference step) on all host cores."""
    ENVS_PER_PROC = 16

    def __init__(self, preset, seed=1234, procs=None):
        import multiprocessing as mp
        self.procs = procs or max(1, min(os.cpu_count() or 1, 32))
        ctx = mp.get_context("spawn")
        self.pool = ctx.Pool(self.procs, initializer=_cpu_init,
                             initargs=(preset, self.ENVS_PER_PROC, seed, ctx.Value("i", 0)))
        self.advance(1)                                   # imports + first step out of the way

    def advance(self, inner):
        """One bench step: every worker advances its envs by `inner` env steps.  Returns wall seconds."""
        t0 = time.perf_counter()
        self.pool.map(_cpu_advance, [inner] * self.procs, chunksize=1)
        return time.perf_counter() - t0

    def env_steps(self, inner):
        return self.procs * self.ENVS_PER_PROC * inner

    def close(self):
        self.pool.close(); self.pool.join()


def cpu_baseline_sample(preset, budget_s=15.0):
    arm = CpuOracleArm(preset)
    t1 = arm.advance(1)
    inner = int(max(2, min(200, budget_s / max(t1, 1e-3))))
    wall = arm.advance(inner)
    v = arm.env_steps(inner) / wall
    arm.close()
    return {"value": v, "unit": UNIT, "cores": arm.procs, "kind": "port",
            "sample": f"{arm.procs} processes x {arm.ENVS_PER_PROC} envs x {inner} env steps of the same scenario "
                      f"(numpy float64 oracle port; the reference needs pybullet/PyFlyt, absent here), {wall:.1f} s wall"}


def run_reference_arm(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from dronechase_b200.config import preset as make_preset
    cfg = make_preset(a.preset)
    arm = CpuOracleArm(a.preset, seed=a.seed)
    t1 = arm.advance(1)
    # size one bench step so that warmup + steps stay around 30 s of CPU work
    inner = int(max(1, min(100, 30.0 / max((a.steps + a.warmup) * t1, 1e-3))))
    for _ in range(a.warmup):
        arm.advance(inner)
    t0 = time.perf_counter()
    for _ in range(a.steps):
        arm.advance(inner)
    wall = time.perf_counter() - t0
    arm.close()
    value = arm.env_steps(inner) * a.steps / wall
    sample = (f"{arm.procs} processes x {arm.ENVS_PER_PROC} envs x {inner} env steps per bench step "
              "(numpy float64 oracle port of the reference step)")
    metric = METRIC if cfg.family == "stage03" else f"{a.preset} env-steps/sec"       # same naming as the GPU arm
    line = {"impl": "reference", "metric": metric, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": 1e3 * wall / max(a.steps, 1), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"{cfg.family} {a.preset}: {cfg.n_lw} LW + {cfg.n_lm} LM per env, uniform random actions, auto-reset; "
                                   "CPU oracle port (the reference itself needs pybullet/PyFlyt, absent from this image)",
                       "envs": arm.procs * arm.ENVS_PER_PROC},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": arm.procs, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------- GPU arm
def run_gpu_arm(a):
    import torch
    import torch.distributed as dist
    from dronechase_b200 import BatchedThreatEngageEnv, _lib, preset as make_preset
    from dronechase_b200.vec_env import DroneChaseVecEnv

    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    # stdout carries exactly ONE JSON line: libraries that print there (NCCL announces its version on stdout) are sent
    # to stderr for the duration of the run
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    cfg = make_preset(a.preset)
    E = a.envs
    strong = a.total_envs > 0
    if strong:
        if a.total_envs % world:
            raise SystemExit("--total-envs must be a multiple of the GPU count")
        E = a.total_envs // world
    dev = torch.device(f"cuda:{local}")
    env = BatchedThreatEngageEnv(cfg, n_envs=E, seed=a.seed, device=local, env_offset=rank * E, auto_reset=True,
                                 sub_batches=a.sub_batches, with_student=a.student)
    env.reset()
    step = env.step
    if a.graph:
        env.capture_step_graphs()
        step = env.step_graph
    # a bank of pre-drawn uniform actions U([-1,-1,-1,0],[1,1,1,1]); each step reads another slab (zero copy)
    gen = torch.Generator(device=dev); gen.manual_seed(a.seed + rank)
    n_bank = 8
    bank = torch.rand(n_bank, E, 4, device=dev, generator=gen)
    bank[..., :3] = bank[..., :3] * 2 - 1
    bank = [bank[i].contiguous() for i in range(n_bank)]

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # spin the scenario up so the timed region sees a realistic mix of waves/armed drones
    for i in range(a.spinup):
        step(bank[i % n_bank])
    for i in range(a.warmup):
        step(bank[i % n_bank])
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    launches0 = _lib.lib().dc_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for i in range(a.steps):
        step(bank[i % n_bank])
    ev1.record()
    barrier()
    launches = _lib.lib().dc_launch_count() - launches0
    if a.graph:                                   # replays do not pass through the library's launch counter
        launches = a.steps * env.launches_per_graph_step
    ms = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    clocks = sampler.stop() if rank == 0 else None
    if a.dump_outputs and rank == 0:
        # step and step_graph return these buffers of the env: they hold the last timed step's outputs until the next step
        dump_outputs(a.dump_outputs, {**{"obs_" + k: v for k, v in env.obs.items()}, "reward": env.reward, "done": env.done,
                                      "info": env.info}, seed=a.seed)
    ms = float(ms.item())
    armed = float((env.get_state()["armed"]).mean()) if rank == 0 else 0.0
    # the one collective of the path: episode statistics at rollout end
    stats = env.stats.clone()
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.SUM)
    stats = stats.cpu().tolist()

    # ---- end-to-end through the public numpy-facing API (SB3 VecEnv contract), host buffers ----
    e2e = None
    if not a.no_e2e:
        import numpy as np
        Ee = min(E, a.e2e_envs)
        venv = DroneChaseVecEnv(cfg, n_envs=Ee, seed=a.seed, device=local, env_offset=rank * Ee, terminal_observation=True)
        venv.reset()
        rng = np.random.RandomState(a.seed + rank)
        acts = [np.concatenate([rng.uniform(-1, 1, (Ee, 3)), rng.uniform(0, 1, (Ee, 1))], axis=1).astype(np.float32) for _ in range(4)]
        ksteps = max(3, min(a.steps, a.e2e_steps))
        for i in range(3):
            venv.step(acts[i % 4])
        barrier()
        t0 = time.perf_counter()
        for i in range(ksteps):
            venv.step(acts[i % 4])
        torch.cuda.synchronize()
        t_e2e = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
        e2e = {"value": world * Ee * ksteps / float(t_e2e.item()), "unit": UNIT, "h2d_bytes_per_step": venv.h2d_bytes_per_step,
               "d2h_bytes_per_step": venv.d2h_bytes_per_step, "envs_per_gpu": Ee, "steps": ksteps,
               "api": "DroneChaseVecEnv.step (numpy in, numpy obs/reward/done/info out incl. infos[i]['terminal_observation'] of "
                      "the envs that auto-reset; pinned staging)",
               "lidar_transfer": ("change list: dc_diff_hits on the device, (index, value) pairs D2H (the fixed first chunk is in "
                                  "d2h_bytes_per_step), dc_host_apply_pairs on %d host threads" % venv._threads if getattr(venv, "pairs", False)
                                  else "device-mapped host arrays, dc_mirror_hits (a few PCIe words per env; not in d2h_bytes_per_step)"
                                  if venv.mapped else "hit list D2H + host scatter")}
        venv.close()

    # ---- end-to-end with the policy ON the device: DeviceRollout.collect, nothing crosses PCIe (SURVEY 8(f)1) ----
    rollout = None
    if not a.no_rollout and cfg.family != "level5" and not cfg.level5_multi_obs:
        from dronechase_b200.policy import LidarInertialActionPolicy
        from dronechase_b200.rollout import DeviceRollout
        Er = min(E, a.e2e_envs)
        renv = BatchedThreatEngageEnv(cfg, n_envs=Er, seed=a.seed, device=local, env_offset=rank * Er, auto_reset=True, with_hits=True)
        renv.reset()
        T = 16
        ro = DeviceRollout(renv, n_steps=T)
        module = LidarInertialActionPolicy(renv, seed=a.seed)

        def timed_collect(pol):
            ro.collect(pol, n_steps=4)
            barrier()
            r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            r0.record()
            ro.collect(pol)
            r1.record()
            barrier()
            t_ro = torch.tensor([r0.elapsed_time(r1)], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t_ro, op=dist.ReduceOp.MAX)
            return world * Er * T / (float(t_ro.item()) * 1e-3)
        # the policy as ONE hand-written kernel (csrc/policy_kernel.cu): float32-grade 3xTF32 is the headline of this arm,
        # plain TF32 and the torch module (cuDNN / cuBLAS float32) are timed beside it
        fused = module.fused("3xtf32")
        v_fused = timed_collect(fused)
        fast = module.fused("tf32")
        v_fast = timed_collect(fast)
        v_torch = timed_collect(module)
        rollout = {"value": v_fused, "unit": UNIT, "envs_per_gpu": Er, "steps": T,
                   "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "policy": fused.describe(),
                   "policy_tf32": {"value": v_fast, "unit": UNIT, "note": "same kernel, plain TF32 operands (actions within 5e-3 of float32)"},
                   "policy_torch_module": {"value": v_torch, "unit": UNIT, "note": "the same network as torch.nn modules (cuDNN / cuBLAS float32)"},
                   "api": "DeviceRollout.collect(policy.fused()): observation -> dc_policy_forward (one kernel: conv + MLPs + pi + action_net) "
                          "-> action -> dc_step, all in HBM; the rollout keeps the sphere as its hit list"}
        fused.close(); fast.close()
        renv.close()

    # ---- the sibling stage03 preset, short (the headline above is a.preset) ----
    also = None
    sibling = {"exp02_v2_full": "exp02_vFinal", "exp02_vFinal": "exp02_v2_full"}.get(a.preset)
    if sibling and not a.no_also and not a.graph:
        env.close()
        env2 = BatchedThreatEngageEnv(make_preset(sibling), n_envs=E, seed=a.seed, device=local, env_offset=rank * E, auto_reset=True,
                                      sub_batches=a.sub_batches)
        env2.reset()
        for i in range(a.spinup + a.warmup):
            env2.step(bank[i % n_bank])
        barrier()
        s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n2 = max(10, min(a.steps, 100))
        s0.record()
        for i in range(n2):
            env2.step(bank[i % n_bank])
        s1.record()
        barrier()
        t2 = torch.tensor([s0.elapsed_time(s1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t2, op=dist.ReduceOp.MAX)
        also = {sibling: {"value": world * E * n2 / (float(t2.item()) * 1e-3), "unit": UNIT, "ms_per_step": float(t2.item()) / n2,
                          "steps": n2, "envs_per_gpu": E}}
        env2.close()

    if rank == 0:
        value = world * E * a.steps / (ms * 1e-3)
        level5 = cfg.family == "level5"
        B = algorithmic_bytes_level5(cfg.n_lw, cfg.n_lm, cfg.level5_multi_obs, a.student) if level5 else algorithmic_bytes_per_env_step(cfg.n_lw, cfg.n_lm, cfg.lidar_channels)
        obs_desc = "(6,3,13,26)+mask 6+15+4" if level5 else f"({cfg.lidar_channels},13,26)+15+4"
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
        else:
            peak, peak_src = 6650.0, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"
        kernel_ms = ms / a.steps                       # two launches per step, events on the launching stream
        achieved = B * E / (kernel_ms * 1e-3) / 1e9
        traffic = warp_inst = None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            cap = json.load(open(tpath)).get(f"{a.preset}@{E}", {})        # ncu capture of this workload only
            traffic, warp_inst = cap.get("dram_bytes_per_launch"), cap.get("warp_instructions_per_step")
        # the two honest views next to the nominal HBM one: DRAM bytes the kernels really move (ncu) over the same time,
        # and the issue-slot floor -- executed warp instructions / (SMs x 4 schedulers x SM clock) over the step time
        n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
        sm_hz = 1e6 * float((clocks or {}).get("sm_mhz") or 1965)
        frac_measured = (traffic / (kernel_ms * 1e-3) / 1e9 / peak) if traffic else None
        issue_frac = (warp_inst / (n_sm * 4 * sm_hz) / (kernel_ms * 1e-3)) if warp_inst else None
        cpu = None
        if world == 1 and not a.no_cpu:
            cpu = cpu_baseline_sample(a.preset)
        metric = METRIC if cfg.family == "stage03" else f"{a.preset} env-steps/sec"
        line = {"metric": metric, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
                "ms_per_step": kernel_ms, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic",
                "config": {"workload": f"{cfg.family} {a.preset}: {cfg.n_lw} LW + {cfg.n_lm} LM per env, {E} envs per GPU, "
                                       f"uniform random actions, auto-reset, obs {obs_desc}",
                           "envs_per_gpu": E, "total_envs": world * E,
                           "parallelism": f"env-sharded x{world}, no step-path collective" + (" (strong scaling: --total-envs)" if strong else ""),
                           "cache": f"inputs larger than L2: {E * B / 1e6:.0f} MB touched per step vs 126 MB L2",
                           "armed_fraction": armed, "spinup_steps": a.spinup,
                           **({"student_observation": "second stacked observation per step (stack_kernel<STUDENT>)"} if a.student else {}),
                           "sub_batches": (a.sub_batches or ("automatic (dc_config.sub_batches = 0): 2 streams from 32,768 envs" if E >= 32768 else 1)),
                           "stepping": ("two captured CUDA graphs replayed alternately (step_graph); actions copied into the bound buffer each step"
                                        if a.graph else "dc_step per step, zero-copy actions")},
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": traffic, "frac_on_measured_bytes": frac_measured, "issue_frac": issue_frac,
                             "warp_instructions_per_step": warp_inst, "algorithmic_bytes_per_env_step": B, "peak_source": peak_src,
                             "kernel": ("dyn_kernel<float,noise> + env_kernel<float,STEP>" + (" + stack_kernel<float>" if level5 else "")
                                        + " (the launches of one env step, timed together; sub-batches overlap them)"),
                             "note": "frac = nominal (SURVEY 8(d) algorithmic bytes: full state + full observation rewrite per env step); "
                                     "the kernels move far fewer bytes (only armed drones are touched, spheres are maintained "
                                     "incrementally): frac_on_measured_bytes is the DRAM view, issue_frac the bound that binds -- "
                                     "the step is instruction-issue / latency bound, not HBM bound"},
                "gpu_launches": int(launches), "clocks": clocks, "e2e": e2e, "e2e_device_rollout": rollout, "also": also,
                "episode_stats": {"episodes": stats[0], "mean_return": stats[1] / max(stats[0], 1), "mean_length": stats[2] / max(stats[0], 1),
                                  "agent_kills": stats[3], "deads": stats[5]}}
        if cpu is not None:
            line["cpu_baseline"] = cpu
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------- LiDAR microbenchmark
def run_lidar_bench(a):
    """BASELINE config 4: threatsense projection LiDAR, 16 entities per env (6 wingmen + 10 munitions), every
    wingman observes -> 6 spheres (3,13,26) per env.  One step = dc_lidar_project over all envs."""
    import numpy as np
    import torch
    from dronechase_b200 import _lib, lidar_project
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device")
    dev = torch.device("cuda:0")
    E, N, O = a.envs if a.envs != 65536 else 16384, 16, 6
    gen = torch.Generator(device=dev); gen.manual_seed(a.seed)
    direction = torch.randn(E, N, 3, device=dev, generator=gen)
    radius = 6.0 * torch.rand(E, N, 1, device=dev, generator=gen) ** (1.0 / 3.0)
    pos = (direction / direction.norm(dim=-1, keepdim=True) * radius).contiguous()
    quat = torch.randn(E, N, 4, device=dev, generator=gen)
    quat = (quat / quat.norm(dim=-1, keepdim=True)).contiguous()
    types = torch.tensor([3] * O + [1] * (N - O), dtype=torch.int32)
    alive = torch.ones(E, N, dtype=torch.uint8, device=dev)
    obs_slot = torch.arange(O, dtype=torch.int32)
    out = torch.empty(E, O, 3, 13, 26, dtype=torch.float32, device=dev)
    types_d, obs_d = types.to(dev), obs_slot.to(dev)
    for _ in range(max(a.warmup, 3)):
        lidar_project(pos, quat, types_d, alive, obs_d, "fused", 40.0, out=out)
    torch.cuda.synchronize()
    sampler = ClockSampler(0); sampler.start(); time.sleep(0.3)
    l0 = _lib.lib().dc_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(a.steps):
        lidar_project(pos, quat, types_d, alive, obs_d, "fused", 40.0, out=out)
    ev1.record(); torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1) / a.steps
    launches = _lib.lib().dc_launch_count() - l0
    clocks = sampler.stop()
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, {"spheres": out}, seed=a.seed)
    spheres = E * O
    # end to end: host positions/quaternions in (pinned), spheres out (pinned)
    h_pos, h_quat = pos.cpu().pin_memory(), quat.cpu().pin_memory()
    h_out = torch.empty(out.shape, dtype=torch.float32).pin_memory()
    ks = max(3, min(a.steps, 20))
    t0 = time.perf_counter()
    for _ in range(ks):
        pos.copy_(h_pos, non_blocking=True); quat.copy_(h_quat, non_blocking=True)
        lidar_project(pos, quat, types_d, alive, obs_d, "fused", 40.0, out=out)
        h_out.copy_(out, non_blocking=True)
        torch.cuda.synchronize()
    e2e_v = spheres * ks / (time.perf_counter() - t0)
    # CPU baseline: the oracle's projection on a bounded sample, one core
    from oracle.env_oracle import lidar_project as oracle_project
    p_np, q_np = pos[:64].cpu().numpy(), quat[:64].cpu().numpy().astype(np.float64)
    t0 = time.perf_counter(); n_cpu = 0
    for e in range(64):
        for o in range(O):
            others = [k for k in range(N) if k != o]
            oracle_project(p_np[e, o], q_np[e, o], p_np[e, others], types.numpy()[others], others, "fused", 40.0)
            n_cpu += 1
    cpu_v = n_cpu / (time.perf_counter() - t0)
    B = 4632
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak = float(json.load(open(peaks_path))["hbm_gbs"]) if os.path.exists(peaks_path) else 6650.0
    achieved = B * spheres / (ms * 1e-3) / 1e9
    line = {"metric": "threatsense LiDAR spheres/sec", "value": spheres / (ms * 1e-3), "unit": "spheres/s", "n_gpus": 1,
            "steps": a.steps, "warmup": max(a.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64 projection on f32 snapshots", "data": "synthetic",
            "config": {"workload": f"projection LiDAR 13x26x3, {N} entities/env ({O} observing wingmen), {E} envs -> {spheres} spheres/step",
                       "cache": f"output {spheres * 4056 / 1e6:.0f} MB per step vs 126 MB L2"},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                         "algorithmic_bytes_per_sphere": B, "kernel": "lidar_kernel"},
            "gpu_launches": int(launches), "clocks": clocks,
            "e2e": {"value": e2e_v, "unit": "spheres/s", "h2d_bytes_per_step": int(h_pos.numel() * 4 + h_quat.numel() * 4),
                    "d2h_bytes_per_step": int(h_out.numel() * 4)},
            "cpu_baseline": {"value": cpu_v, "unit": "spheres/s", "cores": 1, "kind": "port",
                             "sample": f"{n_cpu} spheres through oracle.env_oracle.lidar_project (numpy float64)"}}
    print(json.dumps(line), flush=True)


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--workload", default="env", choices=["env", "lidar"])
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=200)
    p.add_argument("--warmup", type=int, default=5)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--envs", type=int, default=65536, help="envs per GPU (weak scaling)")
    p.add_argument("--total-envs", type=int, default=0,
                   help="STRONG scaling: this many envs in total, sharded over the GPUs (BASELINE config 3 is 65,536 over 8)")
    p.add_argument("--preset", default="exp02_v2_full",
                   help="exp02_v2_full = BASELINE's 'stage03 full scenario with active invaders and protected area'")
    p.add_argument("--no-also", action="store_true", help="skip the short second measurement of the sibling stage03 preset")
    p.add_argument("--no-rollout", action="store_true", help="skip the device-resident rollout arm (policy inference on the GPU)")
    p.add_argument("--sub-batches", type=int, default=0, help="dc_config.sub_batches (0 = automatic)")
    p.add_argument("--graph", action="store_true", help="step through the captured CUDA graphs (BatchedThreatEngageEnv.step_graph)")
    p.add_argument("--student", action="store_true",
                   help="level5_fusion: also build info['student_observation'] (second stack per step, dc_buffers.student_*)")
    p.add_argument("--seed", type=int, default=1234)
    p.add_argument("--spinup", type=int, default=150, help="untimed steps before warm-up so waves/occupancy settle")
    p.add_argument("--e2e-envs", type=int, default=65536)
    p.add_argument("--e2e-steps", type=int, default=30)
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-cpu", action="store_true")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="write the outputs of the last timed step as DIR/<name>.npy (float32 / float64; a fixed, seeded "
                        "sample of envs when all of them would pass 48 MB)")
    a = p.parse_args()
    if a.steps < 1:
        p.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        p.error("--dump-outputs records the GPU path; the reference arm has no outputs to write")
    if a.impl == "reference":
        return run_reference_arm(a)
    if a.workload == "lidar":
        return run_lidar_bench(a)
    if a.warmup < 3:
        a.warmup = 3
    run_gpu_arm(a)


if __name__ == "__main__":
    main()

"""``BatchedThreatEngageEnv`` -- torch-tensor front end of the stage03 simulator.

One instance stands for ``n_envs`` copies of the reference's
``threatengage.environments.level4.exp02_vFinal_environment.Exp02vFinalEnvironment`` (or its
exp03/exp04/exp02_v2_full siblings), i.e. for what ``ReinforcementLearningPipeline.
create_vectorized_environment`` builds as ``SubprocVecEnv([...] * n_envs)``
(src/core/rl_framework/utils/pipeline.py:32-61).  ``reset``/``step`` keep the gymnasium semantics
of ``Env.reset`` / ``Env.step`` (exp02_vFinal_environment.py:133-188) for every env at once; all
tensors stay on the device and PyTorch only provides memory and streams.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional

import numpy as np
import torch

from . import _lib
from .config import TaskConfig, preset, quad_param_vector

_NAV = {"air": 0, "full": 1}
_ALLY = {"bt": 0, "stop": 1}
_REWARD = {"vfinal": 0, "v2full": 1, "l5_fusion": 2}
_LIDAR = {"fused": 0, "classic": 1, "raycast": 2}
_DRIVER = {"legacy": 0, "nn": 1, "bt": 2, "stop": 3, "nn_ally": 4}
INFO_KEYS = ("agent_kills", "allies_kills", "deads", "current_wave", "building_life", "step", "max_step",
             "episode_steps")


def carve_outputs(E: int, device, pin: bool = False):
    """One uint8 buffer holding inertial_data [E,15] f32 | last_action [E,4] f32 | reward [E] f32 | info [E,8] i32 | done [E] u8
    back to back (every piece starts 16-byte aligned for any E), and the typed views of it."""
    sizes = (("inertial_data", torch.float32, (E, 15)), ("last_action", torch.float32, (E, 4)), ("reward", torch.float32, (E,)),
             ("info", torch.int32, (E, _lib.DC_INFO_WORDS)), ("done", torch.uint8, (E,)))
    offs, total = {}, 0
    for name, dt, shape in sizes:
        offs[name] = total
        n = int(np.prod(shape)) * torch.empty((), dtype=dt).element_size()
        total += (n + 15) & ~15
    arena = torch.zeros(total, dtype=torch.uint8, pin_memory=True) if pin else torch.zeros(total, dtype=torch.uint8, device=device)
    views = {}
    for name, dt, shape in sizes:
        n = int(np.prod(shape)) * torch.empty((), dtype=dt).element_size()
        views[name] = arena[offs[name]:offs[name] + n].view(dt).view(*shape)
    return arena, views


class BatchedThreatEngageEnv:
    def __init__(self, cfg: TaskConfig | str = "exp02_vFinal", n_envs: int = 1, seed: int = 0,
                 device: int | str | torch.device = 0, env_offset: int = 0, auto_reset: bool = True,
                 precision: str = "f32", with_ids: bool = False, with_terminal_obs: bool = False, with_hits: bool = False,
                 sub_batches: int = 0, with_student: bool = False):
        if isinstance(cfg, str):
            cfg = preset(cfg)
        if cfg.lidar == "raycast" and with_hits:
            raise ValueError("with_hits: the hit list holds one (cell, r_n) per drone slot and cannot describe a ray-cast sphere, "
                             "whose bounding spheres cover several cells (hit-list storage of ray-cast spheres is not built)")
        if not torch.cuda.is_available():
            raise _lib.DroneChaseError("dronechase_b200 needs a CUDA device: there is no CPU fallback")
        self.cfg, self.n_envs, self.seed = cfg, int(n_envs), int(seed)
        self.device = torch.device(device if not isinstance(device, int) else f"cuda:{device}")
        self.precision = precision
        self._L = _lib.lib()
        c = _lib.dc_config()
        c.abi_version = _lib.DC_ABI_VERSION
        c.n_envs, c.n_lw, c.n_lm = self.n_envs, cfg.n_lw, cfg.n_lm
        c.munition, c.step_increment, c.max_step = cfg.munition, cfg.step_increment, cfg.max_step
        c.initial_round, c.substeps = cfg.initial_round, cfg.substeps
        c.lm_nav, c.ally_mode, c.reward, c.lidar = _NAV[cfg.lm_nav], _ALLY[cfg.ally_mode], _REWARD[cfg.reward], _LIDAR[cfg.lidar]
        c.fixed_lw_spawn, c.auto_reset = int(cfg.fixed_lw_spawn), int(auto_reset)
        c.precision = {"f32": 0, "f64": 1}[precision]
        c.env_offset, c.seed = int(env_offset), self.seed
        c.dome_radius, c.born_radius, c.lw_spawn_radius = cfg.dome_radius, cfg.born_radius, cfg.lw_spawn_radius
        c.explosion_range, c.shoot_range, c.cooldown_steps = cfg.explosion_range, cfg.shoot_range, cfg.cooldown_steps
        c.fire_probability, c.lm_speed, c.bt_speed = cfg.fire_probability, cfg.lm_speed, cfg.bt_speed
        c.ally_stop_mag, c.vel_bonus = cfg.ally_stop_mag, cfg.vel_bonus
        c.building = (C.c_double * 3)(*cfg.building)
        c.quad = (C.c_double * _lib.DC_QUAD_PARAM_WORDS)(*quad_param_vector(cfg.model, cfg.noise_ratio, cfg.gyro_term, cfg.ground_z))
        c.family = {"stage03": 0, "stage02": 1, "stage01": 2, "level5": 3}[cfg.family]
        c.initial_invaders, c.invaders_per_round, c.max_rounds = cfg.initial_invaders, cfg.invaders_per_round, cfg.max_rounds
        c.support_munition = cfg.support_munition
        c.respawn_r_min, c.respawn_r_max = cfg.respawn_r
        c.level5_base_env = int(cfg.level5_base_env)
        c.level5_multi_obs = int(cfg.level5_multi_obs)
        c.sub_batches = int(sub_batches)      # 0 = automatic (dc_config.sub_batches)
        c.lw_driver = (C.c_int32 * 8)(*([_DRIVER[d] for d in cfg.lw_driver] + [0] * (8 - len(cfg.lw_driver))))
        c.eval_task, c.time_is_limited = int(cfg.eval_task), int(cfg.time_is_limited)
        self._c = c
        self._sim = C.c_void_p()
        _lib.check(self._L.dc_create(C.byref(c), self.device.index or 0, C.byref(self._sim)), "dc_create")
        if cfg.lidar == "raycast":
            _lib.check(self._L.dc_set_ray_radii(self._sim, *cfg.ray_radius), "dc_set_ray_radii")
        E, dev = self.n_envs, self.device
        f32 = dict(dtype=torch.float32, device=dev)
        self.actions = torch.zeros(E, 4, **f32)
        level5 = cfg.family == "level5"
        if level5:      # Level5C1FusionEnvironment.compute_observation (level5_c1_fusion_environment.py:47-57)
            lidar_key, lidar = "stacked_spheres", torch.ones(E, _lib.DC_LIDAR_STACK, 3, _lib.N_THETA, _lib.N_PHI, **f32)
        else:
            lidar_key, lidar = "lidar", torch.ones(E, cfg.lidar_channels, _lib.N_THETA, _lib.N_PHI, **f32)
        # The small per-step outputs live back to back in ONE allocation (`out_arena`, layout `OUT_LAYOUT`): a host adapter
        # fetches them with a single device-to-host copy instead of five (each copy costs ~8 us of latency on the stream)
        self.out_arena, views = carve_outputs(E, dev)
        self.obs: Dict[str, torch.Tensor] = {
            lidar_key: lidar,
            "inertial_data": views["inertial_data"],
            "last_action": views["last_action"],
        }
        if level5:
            self.obs["validity_mask"] = torch.zeros(E, _lib.DC_LIDAR_STACK, dtype=torch.bool, device=dev)
        self.reward, self.done, self.info = views["reward"], views["done"], views["info"]
        self.lidar_ids = torch.full((E, _lib.N_THETA, _lib.N_PHI), -1, dtype=torch.int32, device=dev) if with_ids else None
        self.terminal_obs = ({"inertial_data": torch.zeros(E, 15, **f32), "last_action": torch.zeros(E, 4, **f32)}
                             if with_terminal_obs else None)
        self.stats = torch.zeros(8, dtype=torch.float64, device=dev)
        # sparse description of obs["lidar"]: per entity slot (cell, float bits of r_n) or cell = -1 (dc_buffers.lidar_hits)
        # (level5: the hit list of the stacked observation, [E, 5 D + 1, 2], -1 terminated)
        self.lidar_hits = (torch.full((E, 5 * cfg.n_drones + 1 if level5 else cfg.n_drones, 2), -1, dtype=torch.int32, device=dev)
                           if with_hits else None)
        # info["student_observation"] of the base Level5Environment (level5_envrionment.py:291-292,342-346): the second
        # compute_observation call of every step / reset -- same ring, own fusion draws (dc_buffers.student_*)
        self.student_obs = None
        self.student_hits = None
        if with_student:
            if not (level5 and cfg.level5_base_env):
                raise ValueError("with_student needs a level5 preset with level5_base_env (Level5FusionEnvironment)")
            self.student_obs = {
                "stacked_spheres": torch.ones(E, _lib.DC_LIDAR_STACK, 3, _lib.N_THETA, _lib.N_PHI, **f32),
                "validity_mask": torch.zeros(E, _lib.DC_LIDAR_STACK, dtype=torch.bool, device=dev),
                "inertial_data": self.obs["inertial_data"], "last_action": self.obs["last_action"]}
            if with_hits:
                self.student_hits = torch.full((E, 5 * cfg.n_drones + 1, 2), -1, dtype=torch.int32, device=dev)
        # Level5DumbMultiObs.compute_info (level5_dumb_multiobs.py:112-150): one student observation + teacher action per
        # wingman slot; rows with present == 0 (disarmed wingmen) are not in the reference's lists (dc_buffers.mo_*)
        self.multi_obs = None
        self.multi_hits = None
        if level5 and cfg.level5_multi_obs == 1:
            L = cfg.n_lw
            self.multi_obs = {
                "stacked_spheres": torch.ones(E, L, _lib.DC_LIDAR_STACK, 3, _lib.N_THETA, _lib.N_PHI, **f32),
                "validity_mask": torch.zeros(E, L, _lib.DC_LIDAR_STACK, dtype=torch.bool, device=dev),
                "inertial_data": torch.zeros(E, L, 15, **f32),
                "last_action": torch.zeros(E, L, 4, **f32),           # == info["teacher_actions"]
                "present": torch.zeros(E, L, dtype=torch.bool, device=dev)}
            if with_hits:
                self.multi_hits = torch.full((E, L, 5 * cfg.n_drones + 1, 2), -1, dtype=torch.int32, device=dev)
        # wingmen flown by policies inside the task (exp05, level4 evaluation): what compute_lw_observation hands to the
        # policies (dc_lw_observe) and the actions they return (dc_buffers.lw_*), one row per wingman slot
        self.lw_obs = None
        self.lw_actions = self.lw_info = None
        if cfg.lw_driver or cfg.eval_task:
            L = cfg.n_lw
            self.lw_info = torch.zeros(E, L, 4, dtype=torch.int32, device=dev)      # lw_kills, armed, lw_munitions, 0
            if cfg.policy_slots:
                self.lw_obs = {"lidar": torch.ones(E, L, 3, _lib.N_THETA, _lib.N_PHI, **f32),
                               "inertial_data": torch.zeros(E, L, 15, **f32),
                               "present": torch.zeros(E, L, dtype=torch.bool, device=dev)}
                self.lw_actions = torch.zeros(E, L, 4, **f32)
        b = _lib.dc_buffers()
        b.actions, b.obs_lidar = self.actions.data_ptr(), self.obs[lidar_key].data_ptr()
        if self.lw_info is not None:
            b.lw_info = self.lw_info.data_ptr()
        if self.lw_obs is not None:
            b.lw_actions, b.lw_lidar = self.lw_actions.data_ptr(), self.lw_obs["lidar"].data_ptr()
            b.lw_inertial, b.lw_present = self.lw_obs["inertial_data"].data_ptr(), self.lw_obs["present"].data_ptr()
        if level5:
            b.obs_mask = self.obs["validity_mask"].data_ptr()
        b.obs_inertial, b.obs_last_action = self.obs["inertial_data"].data_ptr(), self.obs["last_action"].data_ptr()
        b.reward, b.done, b.info = self.reward.data_ptr(), self.done.data_ptr(), self.info.data_ptr()
        b.lidar_ids = self.lidar_ids.data_ptr() if with_ids else None
        if with_terminal_obs:
            b.term_inertial = self.terminal_obs["inertial_data"].data_ptr()
            b.term_last_action = self.terminal_obs["last_action"].data_ptr()
        b.stats = self.stats.data_ptr()
        if self.lidar_hits is not None:
            b.lidar_hits = self.lidar_hits.data_ptr()
        if self.student_obs is not None:
            b.student_lidar = self.student_obs["stacked_spheres"].data_ptr()
            b.student_mask = self.student_obs["validity_mask"].data_ptr()
            if self.student_hits is not None:
                b.student_hits = self.student_hits.data_ptr()
        if self.multi_obs is not None:
            m = self.multi_obs
            b.mo_lidar, b.mo_mask = m["stacked_spheres"].data_ptr(), m["validity_mask"].data_ptr()
            b.mo_inertial, b.mo_last_action = m["inertial_data"].data_ptr(), m["last_action"].data_ptr()
            b.mo_present = m["present"].data_ptr()
            if self.multi_hits is not None:
                b.mo_hits = self.multi_hits.data_ptr()
        self._b = b
        _lib.check(self._L.dc_bind(self._sim, C.byref(b)), "dc_bind")
        self.steps_done = 0

    @property
    def env_offset(self) -> int:
        """Global index of this env batch's first env (dc_config.env_offset): the env coordinate of its random streams."""
        return int(self._c.env_offset)

    # ------------------------------------------------------------------ gym-like API
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def reset(self, mask: Optional[torch.Tensor] = None):
        """Env.reset for all envs (or those with mask != 0).  Returns the observation dict."""
        ptr = None
        if mask is not None:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
            ptr = C.c_void_p(mask.data_ptr())
        with torch.cuda.device(self.device):
            _lib.check(self._L.dc_reset(self._sim, ptr, self._stream()), "dc_reset")
        return self.obs

    def lw_observe(self) -> Dict[str, torch.Tensor]:
        """First phase of a step with policy-driven wingmen (dc_lw_observe): ``lidar`` [E,n_lw,3,13,26], ``inertial_data``
        [E,n_lw,15], ``present`` [E,n_lw] -- rows of the slots in ``cfg.policy_slots``.  The policies' float32 actions go into
        ``self.lw_actions[:, slot]`` before ``step``; dronechase_b200.drivers.TaskDrivers does the whole loop."""
        if self.lw_obs is None:
            raise _lib.DroneChaseError("this preset has no policy-driven wingman (TaskConfig.lw_driver)")
        with torch.cuda.device(self.device):
            _lib.check(self._L.dc_lw_observe(self._sim, self._stream()), "dc_lw_observe")
        return self.lw_obs

    def step(self, actions: Optional[torch.Tensor] = None):
        """Env.step for all envs: (obs dict, reward[E], terminated[E] uint8, info[E,8] int32)."""
        if actions is not None:
            if (actions.is_cuda and actions.dtype == torch.float32 and actions.is_contiguous()
                    and tuple(actions.shape) == (self.n_envs, 4) and actions.data_ptr() % 16 == 0):
                self._keep = actions                       # zero copy: the kernel reads the policy's tensor
                _lib.check(self._L.dc_set_actions(self._sim, C.c_void_p(actions.data_ptr())), "dc_set_actions")
            else:
                self.actions.copy_(actions, non_blocking=True)
                _lib.check(self._L.dc_set_actions(self._sim, C.c_void_p(self.actions.data_ptr())), "dc_set_actions")
        with torch.cuda.device(self.device):
            _lib.check(self._L.dc_step(self._sim, self._stream()), "dc_step")
        if getattr(self, "_graphs", None) is not None:
            self._graph_next ^= 1                          # the library's parity moved: keep the graph pair in step
        self.steps_done += 1
        return self.obs, self.reward, self.done, self.info

    # ------------------------------------------------------------------ CUDA-graph stepping
    def capture_step_graphs(self):
        """Capture dc_step (all sub-batches, their fork/join events included) into two CUDA graphs, one per step parity
        (the library ping-pongs its snapshot/work-list buffers, and the parity is a kernel argument).  The graphs read
        the actions from ``self.actions``; ``step_graph`` copies the policy's tensor there and replays.  Nothing is
        executed by the capture and the env state is untouched.  Worth it when the step is launch-bound: four
        sub-batches cost eight launches and eight event operations per step, one graph launch replaces them."""
        _lib.check(self._L.dc_set_actions(self._sim, C.c_void_p(self.actions.data_ptr())), "dc_set_actions")
        self._graphs = []
        n0 = self._L.dc_launch_count()
        with torch.cuda.device(self.device):
            torch.cuda.synchronize(self.device)
            for _ in range(2):
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    _lib.check(self._L.dc_step(self._sim, self._stream()), "dc_step (capture)")
                self._graphs.append(g)
        self._graph_next = 0
        self.launches_per_graph_step = int(self._L.dc_launch_count() - n0) // 2     # kernels one replay launches
        return self

    def step_graph(self, actions: Optional[torch.Tensor] = None):
        """Env.step through the captured graphs (same results as ``step``, bit for bit)."""
        if getattr(self, "_graphs", None) is None:
            self.capture_step_graphs()
        if actions is not None:
            self.actions.copy_(actions, non_blocking=True)
        self._graphs[self._graph_next].replay()
        _lib.check(self._L.dc_note_graph_replay(self._sim), "dc_note_graph_replay")
        self._graph_next ^= 1
        self.steps_done += 1
        return self.obs, self.reward, self.done, self.info

    def info_dict(self) -> Dict[str, torch.Tensor]:
        return {k: self.info[:, i] for i, k in enumerate(INFO_KEYS)}

    def close(self):
        if getattr(self, "_sim", None) is not None and self._sim.value:
            self._L.dc_destroy(self._sim)
            self._sim = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------------ parity harness
    def _copy(self, which: int, arr: np.ndarray, to_device: bool):
        assert arr.flags["C_CONTIGUOUS"] and arr.nbytes == self._L.dc_state_bytes(self._sim, which)
        _lib.check(self._L.dc_copy_state(self._sim, which, arr.ctypes.data_as(C.c_void_p), arr.nbytes, int(to_device)),
                   "dc_copy_state")

    def get_state(self) -> Dict[str, np.ndarray]:
        """Decode the raw device state (layout in include/dronechase_b200.h) into named arrays."""
        E, D = self.n_envs, self.cfg.n_drones
        rt = np.float64 if self.precision == "f64" else np.float32
        raw = np.empty((_lib.DC_STATE_QUADS, E * D, 4), dtype=rt)
        self._copy(0, raw, False)
        q = raw.reshape(_lib.DC_STATE_QUADS, E, D, 4).astype(np.float64)
        env = np.empty((E, _lib.DC_ENV_WORDS), dtype=np.int32)
        self._copy(1, env, False)
        lw = np.empty((E, self.cfg.n_lw, 3), dtype=np.float64)
        self._copy(2, lw, False)
        flags = q[0, ..., 3].astype(np.int64)
        last_closest = env[:, 10:12].copy().view(np.float64)[:, 0]
        return {
            "pos": q[0, ..., :3], "quat": q[1], "vel": q[2, ..., :3], "omega": q[3, ..., :3], "throttle": q[4],
            "pid": np.concatenate([q[5 + k] for k in range(6)], axis=-1),
            "armed": (flags & 1).astype(bool), "off_armed": (flags & 2).astype(bool), "nav": (flags >> 2) & 3,
            "last_fired": q[11, ..., 3], "ammo": flags >> 8,
            "imu_pos": q[11, ..., :3], "formation": q[12, ..., :3],
            "step": env[:, 0].copy(), "max_step": env[:, 1].copy(), "round": env[:, 2].copy(),
            "agent_kills": env[:, 3].copy(), "allies_kills": env[:, 4].copy(), "deads": env[:, 5].copy(),
            "building_life": env[:, 6].copy(), "hit_ctr": env[:, 7].copy(), "spawn_ctr": env[:, 8].copy(),
            "phys_ctr": env[:, 9].copy(), "last_closest": last_closest, "lw_init": lw,
            "_env_words": env,
        }

    def set_state(self, st: Dict[str, np.ndarray]):
        """Inverse of get_state (every key of get_state except the derived '_env_words' is honoured)."""
        E, D = self.n_envs, self.cfg.n_drones
        rt = np.float64 if self.precision == "f64" else np.float32
        q = np.zeros((_lib.DC_STATE_QUADS, E, D, 4), dtype=np.float64)
        flags = (st["armed"].astype(np.int64) | (st["off_armed"].astype(np.int64) << 1) | (st["nav"].astype(np.int64) << 2)
                 | (np.maximum(st["ammo"], 0).astype(np.int64) << 8))
        q[0, ..., :3], q[0, ..., 3] = st["pos"], flags
        q[1] = st["quat"]
        q[2, ..., :3] = st["vel"]
        q[3, ..., :3] = st["omega"]
        q[4] = st["throttle"]
        for k in range(6):
            q[5 + k] = st["pid"][..., 4 * k:4 * k + 4]
        q[11, ..., :3], q[11, ..., 3] = st["imu_pos"], st["last_fired"]
        q[12, ..., :3] = st["formation"]
        self._copy(0, np.ascontiguousarray(q.reshape(_lib.DC_STATE_QUADS, E * D, 4).astype(rt)), True)
        env = st["_env_words"].copy() if "_env_words" in st else np.zeros((E, _lib.DC_ENV_WORDS), dtype=np.int32)
        for i, k in enumerate(("step", "max_step", "round", "agent_kills", "allies_kills", "deads", "building_life",
                               "hit_ctr", "spawn_ctr", "phys_ctr")):
            env[:, i] = st[k]
        env[:, 10:12] = np.ascontiguousarray(st["last_closest"], dtype=np.float64).reshape(E, 1).view(np.int32)
        env[:, 14] = 1
        self._copy(1, np.ascontiguousarray(env, dtype=np.int32), True)
        self._copy(2, np.ascontiguousarray(st["lw_init"], dtype=np.float64), True)


def lidar_project(pos: torch.Tensor, quat: torch.Tensor, types: torch.Tensor, alive: torch.Tensor,
                  obs_slot: torch.Tensor, flavour: str = "fused", radius: float = 40.0, with_ids: bool = False,
                  out: Optional[torch.Tensor] = None):
    """Stand-alone projection LiDAR (dc_lidar_project): pos [E,N,3] f32, quat [E,N,4] f32 (xyzw),
    types [N] i32, alive [E,N] u8, obs_slot [O] i32 -> sphere [E,O,C,13,26] f32 (+ ids [E,O,13,26])."""
    L = _lib.lib()
    E, N, _ = pos.shape
    O = obs_slot.numel()
    ch = 3 if flavour == "fused" else 2
    dev = pos.device
    pos, quat = pos.contiguous().float(), quat.contiguous().float()
    types, obs_slot = types.to(dev, torch.int32).contiguous(), obs_slot.to(dev, torch.int32).contiguous()
    alive = alive.to(dev, torch.uint8).contiguous()
    sphere = out if out is not None else torch.empty(E, O, ch, _lib.N_THETA, _lib.N_PHI, dtype=torch.float32, device=dev)
    ids = torch.empty(E, O, _lib.N_THETA, _lib.N_PHI, dtype=torch.int32, device=dev) if with_ids else None
    with torch.cuda.device(dev):
        _lib.check(L.dc_lidar_project(pos.data_ptr(), quat.data_ptr(), types.data_ptr(), alive.data_ptr(),
                                      obs_slot.data_ptr(), E, N, O, _LIDAR[flavour], float(radius), sphere.data_ptr(),
                                      ids.data_ptr() if with_ids else None,
                                      C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)), "dc_lidar_project")
    return (sphere, ids) if with_ids else sphere


def lidar_raycast(pos: torch.Tensor, quat: torch.Tensor, radius: torch.Tensor, types: torch.Tensor, alive: torch.Tensor,
                  obs_slot: torch.Tensor, max_range: float = 40.0, with_ids: bool = False, out: Optional[torch.Tensor] = None):
    """Opt-in ray-cast LiDAR (dc_lidar_raycast): like lidar_project plus radius [N] f32 bounding spheres."""
    L = _lib.lib()
    E, N, _ = pos.shape
    O = obs_slot.numel()
    dev = pos.device
    pos, quat = pos.contiguous().float(), quat.contiguous().float()
    radius = radius.to(dev, torch.float32).contiguous()
    types, obs_slot = types.to(dev, torch.int32).contiguous(), obs_slot.to(dev, torch.int32).contiguous()
    alive = alive.to(dev, torch.uint8).contiguous()
    sphere = out if out is not None else torch.empty(E, O, 3, _lib.N_THETA, _lib.N_PHI, dtype=torch.float32, device=dev)
    ids = torch.empty(E, O, _lib.N_THETA, _lib.N_PHI, dtype=torch.int32, device=dev) if with_ids else None
    with torch.cuda.device(dev):
        _lib.check(L.dc_lidar_raycast(pos.data_ptr(), quat.data_ptr(), radius.data_ptr(), types.data_ptr(), alive.data_ptr(),
                                      obs_slot.data_ptr(), E, N, O, float(max_range), sphere.data_ptr(),
                                      ids.data_ptr() if with_ids else None,
                                      C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)), "dc_lidar_raycast")
    return (sphere, ids) if with_ids else sphere

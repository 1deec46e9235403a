"""Scenario configuration of the batched stage03 simulator.

``TaskConfig`` gathers the constants the reference scatters over ``Task.init_constants``
(src/threatengage/environments/level4/components/tasks_management/tasks/exp02_vFinal_task.py:87-111),
``Gun.__init__`` (src/core/entities/quadcopters/components/weapons/gun.py:8-35), the navigators
(loitering_munition_navigator.py:56-60, loyalwingman_navigator.py:33-39) and the env constructor
(exp02_vFinal_environment.py:44-49,84-88,112-115).  ``PRESETS`` names them after the reference's
task/env classes.  ``CF2X`` is the drone model in PyFlyt's yaml schema (motor_params / drag_params /
control_params) so the genuine ``cf2x.yaml`` can be substituted: ``TaskConfig(model=yaml.safe_load(...))``.
"""
from __future__ import annotations

import copy
import math
from dataclasses import dataclass, field

import numpy as np

CF2X = {
    "mass": 0.027,
    "inertia": [1.4e-5, 1.4e-5, 2.17e-5],
    "arm": 0.028,
    "motor_params": {"total_thrust": 0.5886, "thrust_coef": 3.16e-10, "torque_coef": 7.94e-12,
                     "noise_ratio": 0.02, "tau": 0.01},
    "drag_params": {"drag_coef_xyz": 1.0, "drag_area_xyz": 0.004},
    "control_params": {
        "ang_vel": {"kp": [8e-3, 8e-3, 1e-2], "ki": [2.5e-7, 2.5e-7, 1.3e-4], "kd": [1e-4, 1e-4, 0.0], "lim": [1.0, 1.0, 1.0]},
        "ang_pos": {"kp": [2.0, 2.0, 2.0], "ki": [0.0, 0.0, 0.0], "kd": [0.0, 0.0, 0.0], "lim": [3.0, 3.0, 3.0]},
        "lin_vel": {"kp": [0.8, 0.8], "ki": [0.3, 0.3], "kd": [0.5, 0.5], "lim": [0.4, 0.4]},
        "lin_pos": {"kp": [1.0, 1.0], "ki": [0.0, 0.0], "kd": [0.0, 0.0], "lim": [2.0, 2.0]},
        "z_pos": {"kp": 1.0, "ki": 0.0, "kd": 0.0, "lim": 1.0},
        "z_vel": {"kp": 0.15, "ki": 1.0, "kd": 0.015, "lim": 1.0},
    },
}

_PID_ORDER = (("ang_vel", 3), ("ang_pos", 3), ("lin_vel", 2), ("z_vel", 1), ("lin_pos", 2), ("z_pos", 1))
RHO_AIR, GRAVITY, GROUND_Z, PHYSICS_HZ, CONTROL_HZ = 1.225, -9.81, -6.0, 240, 120


def quad_param_vector(model: dict, noise_ratio: float | None = None, gyro_term: bool = False,
                      ground_z: float = GROUND_Z) -> np.ndarray:
    """The 88 doubles of dc_config.quad (layout documented in include/dronechase_b200.h)."""
    mp, dp = model["motor_params"], model["drag_params"]
    noise = mp["noise_ratio"] if noise_ratio is None else noise_ratio
    max_rpm = math.sqrt(mp["total_thrust"] / (4.0 * mp["thrust_coef"]))
    drag_k = 0.5 * RHO_AIR * dp["drag_coef_xyz"] * dp["drag_area_xyz"]
    out = [model["mass"], *model["inertia"], model["arm"], mp["thrust_coef"], mp["torque_coef"], mp["tau"],
           noise, max_rpm, drag_k, 1.0 / PHYSICS_HZ, 1.0 / CONTROL_HZ, float(gyro_term), GRAVITY, float(ground_z)]
    for name, n in _PID_ORDER:
        g = model["control_params"][name]
        for key in ("kp", "ki", "kd", "lim"):
            vals = list(np.broadcast_to(np.asarray(g[key], dtype=np.float64), (n,)))
            out.extend(vals + [0.0] * (3 - n))
    return np.asarray(out, dtype=np.float64)


def calculate_rounds(num_defenders: int, munition_per_defender: int) -> int:
    """exp02_vFinal_task.py:197-225: waves 1..n consume n(n+1)/2 rounds of ammunition."""
    total = num_defenders * munition_per_defender
    return math.ceil((-1 + math.sqrt(1 + 8 * total)) / 2)


@dataclass
class TaskConfig:
    n_lw: int = 1                     # NUM_PURSUERS (slot 0 = RL agent)
    n_lm: int | None = None           # NUM_INVADERS; None -> calculate_rounds(n_lw, munition)
    munition: int = 20
    dome_radius: float = 20.0
    rl_frequency: int = 15
    born_radius: float = 6.0
    lw_spawn_radius: float = 2.0
    explosion_range: float = 0.2
    shoot_range: float = 1.0
    step_increment: int = 100
    max_step: int = 300
    initial_round: int = 1
    cooldown_seconds: float = 4.0
    fire_probability: float = 0.9
    lm_speed: float = 0.4
    bt_speed: float = 0.6
    lm_nav: str = "air"               # "air" | "full"
    ally_mode: str = "bt"             # "bt" | "stop"
    ally_stop_mag: float = 1.0
    reward: str = "vfinal"            # "vfinal" | "v2full" | "l5_fusion" (level5 family: Level5FusionTask.compute_reward)
    vel_bonus: float = 1.0
    building: tuple = (0.0, 0.0, 0.1)
    fixed_lw_spawn: bool = False
    lidar: str = "fused"              # "fused" (3,13,26) | "classic" (2,13,26) | "raycast" (3,13,26, needs ray_radius)
    family: str = "stage03"           # "stage03" (level4 tasks) | "stage02" (level3 L3Stage1) | "stage01" (level2) |
                                      # "level5" (threatsense Level5C1FusionTask: random agent, stacked-sphere fusion)
    initial_invaders: int = 4         # level5: wave k arms min((k-1)*invaders_per_round + initial_invaders, n_lm) munitions
    invaders_per_round: int = 1
    max_rounds: int = 7
    level5_base_env: bool = False     # level5: the base Level5Environment's observation protocol (dc_config.level5_base_env)
    level5_multi_obs: int = 0         # level5: 1 = Level5DumbMultiObs, 2 = Level52BTEvaluationEnvironment (dc_config.level5_multi_obs)
    # stage03 tasks whose wingmen are flown by policies INSIDE the task (dc_config.lw_driver / eval_task / time_is_limited):
    # one entry per wingman -- "legacy" (slot 0 = the env's action, the others ally_mode), "nn" (a policy, whenever armed),
    # "bt" (behaviour tree), "stop" (zero velocity), "nn_ally" (a policy, only behind an armed pursuer: exp05)
    lw_driver: tuple = ()
    eval_task: bool = False           # Evaluation_Task + EvaluationEnvironment (evaluation_task.py, evaluation_environment.py)
    time_is_limited: bool = False     # Evaluation_Task TIME_IS_LIMITED
    support_munition: int = 10        # stage02: Gun() default of the support wingman
    respawn_r: tuple = (2.0, 6.0)     # stage02: disarmed munitions reappear on r in U(2, 6)
    ground_z: float = GROUND_Z        # level2/level3 spawn no plane: NO_GROUND
    noise_ratio: float | None = None  # None -> the model's motor_params.noise_ratio
    gyro_term: bool = False
    model: dict = field(default_factory=lambda: copy.deepcopy(CF2X))
    # lidar="raycast": bounding radius (metres) of every wingman and of every munition, (r_lw, r_lm), that the rays of the
    # agent's sphere are tested against.  No default: the reference's body dimensions (getVisualShapeData) are not known here.
    ray_radius: tuple | None = None

    def __post_init__(self):
        if self.n_lm is None:
            self.n_lm = calculate_rounds(self.n_lw, self.munition)
        if self.lidar == "raycast":
            if self.family != "stage03" or self.lw_driver or self.eval_task:
                raise ValueError("lidar='raycast' is built for the stage03 family without lw_driver / eval_task (the agent's "
                                 "sphere only): not for level5 stacks, stage01/02 or policy-driven wingmen")
            r = self.ray_radius
            if r is None or len(r) != 2:
                raise ValueError("lidar='raycast' needs ray_radius=(r_lw, r_lm), the bounding radius in metres of every wingman "
                                 "and of every munition; there is no default")
            if not all(math.isfinite(float(v)) and float(v) >= 0.0 for v in r):
                raise ValueError(f"ray_radius must be finite and >= 0 metres, got {tuple(r)}")
            self.ray_radius = (float(r[0]), float(r[1]))
        elif self.ray_radius is not None:
            raise ValueError("ray_radius is the bounding radius of lidar='raycast' and means nothing to lidar=%r" % self.lidar)

    @property
    def policy_slots(self) -> tuple:
        """Wingman slots flown by a policy inside the task (their observations come from dc_lw_observe)."""
        return tuple(j for j, d in enumerate(self.lw_driver) if d in ("nn", "nn_ally"))

    @property
    def n_drones(self) -> int:
        return self.n_lw + self.n_lm

    @property
    def lidar_channels(self) -> int:
        return 2 if self.lidar == "classic" else 3

    @property
    def substeps(self) -> int:
        # aggregate_sim_steps = int(ctrl_hz / rl_frequency) control steps of updates_per_step physics steps
        return int(CONTROL_HZ / self.rl_frequency) * (PHYSICS_HZ // CONTROL_HZ)

    @property
    def cooldown_steps(self) -> float:
        return self.cooldown_seconds / (1 / 15)      # gun.py:13,25 hard-codes timestep = 1/15


PRESETS = {
    # threatengage/environments/level4/exp02_vFinal_environment.py + tasks/exp02_vFinal_task.py
    "exp02_vFinal": dict(),
    # exp03_vFinal_environment.py / exp03_vFinal_task.py: agent + behaviour-tree wingman vs 9 munitions
    "exp03_vFinal": dict(n_lw=2),
    # exp04_vFinal_task.py:240-242,467: second wingman parked, velocity bonus x10
    "exp04_vFinal": dict(n_lw=2, ally_mode="stop", ally_stop_mag=1.0, vel_bonus=10.0),
    # tasks/exp02_v2_full_task.py: protected building, cone FSM, born radius 8
    "exp02_v2_full": dict(born_radius=8.0, lm_nav="full", reward="v2full", ally_mode="stop", ally_stop_mag=0.5,
                          fixed_lw_spawn=True),
    # BASELINE.json config 5: 4 wingmen vs 64 munitions, all armed from the first wave
    "swarm": dict(n_lw=4, n_lm=64, initial_round=64),
}
# exp05_vFinal_environment.py / exp05_vFinal_task.py:252-260: exp03 with the second wingman flown by a second policy
# (Exp05vFinalEnvironment.update_model) instead of the behaviour tree
PRESETS["exp05_vFinal"] = dict(n_lw=2, lw_driver=("legacy", "nn_ally"))
NO_GROUND = -1.0e9
# threatengage/environments/level3/pyflyt_level3_environment_v2.py + components/stages.py L3Stage1:
# agent (4 rounds) + idle support wingman vs 5 hovering munitions that respawn, dome 8, 600 steps
PRESETS["stage02"] = dict(family="stage02", n_lw=2, n_lm=5, munition=4, dome_radius=8.0, max_step=600, initial_round=5,
                          born_radius=2.0, lw_spawn_radius=1.0, lm_speed=0.5, ground_z=NO_GROUND)
PRESETS["stage02_10lm"] = dict(PRESETS["stage02"], n_lm=10, initial_round=10)     # BASELINE config 2 scale knob
# threatengage/environments/level2/pyflyt_level2_environment_modified_v2.py: agent + idle wingman vs one munition
# holding position in QuadX mode 7, caught (teleported) at 0.4 m, dome 10, 300 steps, empty guns
PRESETS["stage01"] = dict(family="stage01", n_lw=2, n_lm=1, munition=0, dome_radius=10.0, max_step=300, initial_round=1,
                          ground_z=NO_GROUND)
PRESETS["stage03"] = PRESETS["exp02_vFinal"]
# threatsense/level5/level5_c1_fusion_environment.py + tasks/level5_c1_fusion_task.py:83-111: 2 wingmen (a random one is
# the agent, the other flies the behaviour tree) vs 4 -> 10 munitions (+1 per wave, 7 waves), 49 rounds each, obs =
# stacked spheres (6,3,13,26) + validity mask (6,) + inertial/gun (15,) + the agent's last command (4,)
PRESETS["level5_c1"] = dict(family="level5", n_lw=2, n_lm=10, munition=49, initial_invaders=4, invaders_per_round=1, max_rounds=7)
# tasks/level5_fusion_task.py:81-112 scale (6 wingmen, 5 -> 30 munitions, +5 per wave, 105 rounds) on the C1 task logic
PRESETS["level5_fusion_scale"] = dict(family="level5", n_lw=6, n_lm=30, munition=105, initial_invaders=5, invaders_per_round=5,
                                      max_rounds=6)


# threatsense/level5/level5_fusion_environment.py (= the base Level5Environment, level5_envrionment.py) +
# tasks/level5_fusion_task.py:81-112,448-613: 6 wingmen vs 5 -> 30 munitions (+5 per wave, 6 waves), 105 rounds each, reward with
# reload-distance shaping clipped to +-3000, every wingman updates its LiDAR, three compute_observation calls per step
PRESETS["level5_fusion"] = dict(PRESETS["level5_fusion_scale"], reward="l5_fusion", level5_base_env=True)
# threatsense/level5/level5_dumb_multiobs.py + tasks/level5_dumb_multiobject_task.py:81-107: the data-collection env of
# apps/threatsense_runner/collect_and_save.py -- 7 wingmen all on the behaviour tree vs 5 -> 30 munitions (+1 per wave, 26
# waves), (5 + 30) * 26 // 2 = 455 rounds each; per step every armed wingman's student observation + its last command
PRESETS["level5_dumb_multiobs"] = dict(family="level5", n_lw=7, n_lm=30, munition=455, initial_invaders=5, invaders_per_round=1,
                                       max_rounds=26, reward="l5_fusion", level5_multi_obs=1)
# threatsense/level5/level5_eval_2bt_environment.py + tasks/level5_2bt_evaluation_task.py:82-113 (apps/threatsense_runner/
# evaluation_2bt.py): 2 behaviour-tree wingmen vs 5 -> 30 munitions, MAX_STEP 1300 never incremented, no reward/observation
PRESETS["level5_eval_2bt"] = dict(family="level5", n_lw=2, n_lm=30, munition=455, initial_invaders=5, invaders_per_round=1,
                                  max_rounds=26, max_step=1300, step_increment=0, reward="l5_fusion", level5_multi_obs=2)


def evaluation_preset(configuration: dict, **overrides) -> TaskConfig:
    """Evaluation_Task._process_configuration (evaluation_task.py:89-110): ``configuration["drivers"]`` = one
    ``{"type": "nn" | "bt" | anything else, "name": ..., "path": ...}`` per wingman; ``munition_per_defender``,
    ``ENEMY_BORN_RADIUS``, ``INITIAL_ROUND``, ``STEP_INCREMENT``, ``MAX_STEP``, ``TIME_IS_LIMITED``."""
    types = [str(d.get("type", "")) for d in configuration.get("drivers", [])]
    if not 1 <= len(types) <= 8:
        raise ValueError("configuration['drivers'] must name 1..8 wingmen")
    kw = dict(n_lw=len(types), munition=int(configuration.get("munition_per_defender", 20)),
              born_radius=float(configuration.get("ENEMY_BORN_RADIUS", 6)), initial_round=int(configuration.get("INITIAL_ROUND", 1)),
              step_increment=int(configuration.get("STEP_INCREMENT", 100)), max_step=int(configuration.get("MAX_STEP", 300)),
              time_is_limited=bool(configuration.get("TIME_IS_LIMITED", False)), eval_task=True,
              lw_driver=tuple(t if t in ("nn", "bt") else "stop" for t in types))
    kw.update(overrides)
    return TaskConfig(**kw)


def preset(name: str, **overrides) -> TaskConfig:
    kw = dict(PRESETS[name])
    kw.update(overrides)
    return TaskConfig(**kw)

/*
 * dronechase_b200 -- C ABI of the batched, GPU-resident replacement for the per-step
 * hot path of DaviGuanabara/dronechase's threatengage "level4" (stage03) environments.
 *
 * Nothing like this boundary exists in the reference (it is 100 % Python); every entry
 * point below replaces a group of reference methods and cites them.  Paths are relative
 * to the reference's src/ directory.
 *
 *   one dc_sim        == N x  threatengage/environments/level4/exp02_vFinal_environment.py:30
 *                             (Exp02vFinalEnvironment and its exp03/exp04/exp02_v2_full siblings),
 *                             i.e. what rl_framework/utils/pipeline.py:58-61 builds as
 *                             SubprocVecEnv([lambda: Env(...)] * n_envs)
 *   dc_reset          ==      Env.reset                        exp02_vFinal_environment.py:133-151
 *   dc_step           ==      Env.step                         exp02_vFinal_environment.py:155-188
 *                             (drive, Task.on_step_start, 16 x L4AviarySimulation substeps
 *                              level4_simulation.py:84-98, Task.on_step_middle, compute_info,
 *                              compute_observation :206-234, Task.on_step_end) followed by the
 *                             VecEnv auto-reset of SB3's DummyVecEnv/SubprocVecEnv when enabled
 *   dc_lidar_project  ==      FusedLIDAR.update_data           core/entities/quadcopters/components/sensors/fused_lidar.py:143-217
 *                             LIDAR.update_data                core/entities/quadcopters/components/sensors/lidar.py:263-280
 *   family DC_FAMILY_LEVEL5:  dc_reset / dc_step == Level5Environment.reset / step   threatsense/level5/level5_envrionment.py:203-266
 *                             with Level5C1FusionEnvironment.compute_observation       threatsense/level5/level5_c1_fusion_environment.py:20-57
 *                             (FusedLIDAR.update_data + read_data of every armed wingman, fused_lidar.py:143-269) and
 *                             Level5C1FusionTask                                       .../tasks/level5_c1_fusion_task.py:285-545
 *
 * Conventions: plain pointers and sizes, no C++/torch types.  Every function returns 0 on
 * success or a negative dc_status; dc_last_error() gives a thread-local message.  Functions
 * never synchronise the device (except dc_copy_state, dc_create, dc_destroy), never allocate
 * after dc_create, and enqueue on the caller's stream (pass torch.cuda.current_stream().cuda_stream).
 * A dc_sim belongs to one device and must be driven by one thread at a time.
 */
#ifndef DRONECHASE_B200_H
#define DRONECHASE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DC_ABI_VERSION 9   /* v9: dc_policy_create_ac / dc_policy_act / dc_gae (PPO rollout collection on the device); v8: dc_policy_* (the agent's network as one kernel; dc_config / dc_buffers unchanged); v7: dc_host_register / dc_host_unregister / dc_mirror_hits */

enum dc_status {
    DC_OK = 0,
    DC_ERR_ARG = -1,        /* bad argument / config */
    DC_ERR_CUDA = -2,       /* a CUDA runtime call failed */
    DC_ERR_UNBOUND = -3,    /* dc_step/dc_reset before dc_bind */
    DC_ERR_NO_DEVICE = -4   /* no CUDA device: there is NO CPU fallback */
};

enum { DC_NAV_AIR_COMBAT_ONLY = 0, DC_NAV_FULL = 1 };   /* loitering_munition_navigator(_air_combat_only).py */
enum { DC_ALLY_BEHAVIOR_TREE = 0, DC_ALLY_STOPPED = 1 }; /* loyalwingman_navigator.py / exp04_vFinal_task.py:240-242 */
enum { DC_REWARD_VFINAL = 0, DC_REWARD_V2FULL = 1,      /* exp02_vFinal_task.py:422-568 / exp02_v2_full_task.py */
       DC_REWARD_L5_FUSION = 2 };                        /* level5 family only: level5_fusion_task.py:448-555 instead of the C1 reward */
enum { DC_LIDAR_FUSED = 0, DC_LIDAR_CLASSIC = 1 };       /* (3,13,26) fused_lidar.py / (2,13,26) lidar.py */
enum { DC_PRECISION_F32 = 0, DC_PRECISION_F64 = 1 };     /* arithmetic + state type of the dynamics */
enum { DC_DRIVER_LEGACY = 0,    /* the task's own rule: slot 0 = dc_buffers.actions, the others dc_config.ally_mode */
       DC_DRIVER_NN = 1,        /* dc_buffers.lw_actions[:, j] whenever armed ("nn": driver.predict(compute_lw_observation)) */
       DC_DRIVER_BT = 2,        /* LoyalWingmanBehaviorTree whenever armed ("bt") */
       DC_DRIVER_STOP = 3,      /* pursuer.drive([0,0,0,1]): zero velocity (any other driver type) */
       DC_DRIVER_NN_ALLY = 4 }; /* lw_actions[:, j], but only behind an armed pursuer: get_armed_pursuers()[1:] (exp05) */
enum { DC_FAMILY_STAGE03 = 0,   /* level4 tasks: waves, navigators, exp02_vFinal_task.py & siblings */
       DC_FAMILY_STAGE02 = 1,   /* level3 L3Stage1: hovering munitions that respawn, level3/components/stages.py */
       DC_FAMILY_STAGE01 = 2,   /* level2 pyflyt_level2_environment_modified_v2.py: catch a position-holding munition */
       DC_FAMILY_LEVEL5 = 3 };  /* threatsense/level5/level5_c1_fusion_environment.py + tasks/level5_c1_fusion_task.py:
                                   random agent among the wingmen, stacked-sphere LiDAR fusion (fused_lidar.py:223-326) */
#define DC_LIDAR_STACK 6         /* spheres per stacked observation: n_neighbors_max + 1 (fused_lidar.py:59,307) */

#define DC_LIDAR_THETA 13
#define DC_LIDAR_PHI 26
#define DC_QUAD_PARAM_WORDS 88   /* oracle/dynamics.py QuadParams.flat(): 16 scalars + 6 PIDs x 4 x 3 */
#define DC_INFO_WORDS 8          /* per env: agent_kills, allies_kills, deads, current_wave,
                                    building_life, step, max_step, episode_steps (of the episode that ended) */
#define DC_STATE_QUADS 13        /* per-drone state: 13 x 4 scalars, see dc_copy_state */
#define DC_ENV_WORDS 16          /* per-env scalar block, 32-bit words */

/* One POD for the whole stage03 task family (exp02_vFinal_task.py:87-111 init_constants). */
typedef struct dc_config {
    int32_t abi_version;        /* DC_ABI_VERSION */
    int32_t n_envs;
    int32_t n_lw;               /* NUM_PURSUERS; slot 0 is the RL agent */
    int32_t n_lm;               /* NUM_INVADERS == MAX_NUMBER_OF_ROUNDS */
    int32_t munition;           /* munition_per_defender */
    int32_t step_increment;     /* STEP_INCREMENT */
    int32_t max_step;           /* MAX_STEP */
    int32_t initial_round;      /* INITIAL_ROUND */
    int32_t substeps;           /* aggregate_sim_steps * updates_per_step = 16 */
    int32_t lm_nav;             /* DC_NAV_* */
    int32_t ally_mode;          /* DC_ALLY_* */
    int32_t reward;             /* DC_REWARD_* (also selects the termination variant) */
    int32_t lidar;              /* DC_LIDAR_* */
    int32_t fixed_lw_spawn;     /* exp02_v2_full_task.py replace_pursuers re-uses the init positions */
    int32_t auto_reset;         /* VecEnv semantics: reset finished envs inside dc_step */
    int32_t precision;          /* DC_PRECISION_* */
    int32_t env_offset;         /* global index of env 0 (multi-GPU shards keep one Philox key space) */
    int32_t family;             /* DC_FAMILY_* */
    uint64_t seed;
    double dome_radius, born_radius, lw_spawn_radius, explosion_range, shoot_range;
    double cooldown_steps, fire_probability, lm_speed, bt_speed, ally_stop_mag, vel_bonus;
    double building[3];
    double quad[DC_QUAD_PARAM_WORDS];
    /* stage02 only (threatengage/environments/level3/components/stages.py:118,170-174,370-376) */
    double respawn_r_min, respawn_r_max;   /* disarmed munitions reappear on r in U(min, max) every step */
    int32_t support_munition;              /* Gun() default of the support wingman (gun.py:11) */
    /* level5 only (level5_c1_fusion_task.py:83-90): wave k arms min((k-1)*invaders_per_round + initial_invaders, n_lm) */
    int32_t initial_invaders;
    int32_t invaders_per_round;
    int32_t max_rounds;
    /* The env batch is run as this many independent sub-batches on internal streams (fork/join around the caller's
     * stream inside dc_step/dc_reset), so that the latency-bound env_kernel of one sub-batch runs under the
     * issue-bound dyn_kernel of another.  0 = automatic (2 from 32,768 float32 envs, else 1).  Results do not depend
     * on it: envs are independent and the Philox streams are keyed by the global env index. */
    int32_t sub_batches;
    /* level5 only.  Non-zero = the BASE Level5Environment's observation protocol (level5_envrionment.py:236-346), which
     * Level5FusionEnvironment inherits: every wingman, armed or not, updates its LiDAR (a dead one re-enters the agent's
     * ring as a publisher without a pose), compute_observation runs three times per step and per reset (the observation,
     * info["student_observation"], info["teacher_observation"]: the fusion draws of the returned observation are those
     * of the first call, obs_call advances by 3), a dead agent's stack is empty, and last_action is the env's
     * (zeroed by reset).  Zero = Level5C1FusionEnvironment (level5_c1_fusion_environment.py:20-57). */
    int32_t level5_base_env;
    /* level5 only (ABI v6).  Non-zero = Level5DumbMultiObs + Level5DumbMultiObjectTask (threatsense/level5/
     * level5_dumb_multiobs.py, .../tasks/level5_dumb_multiobject_task.py), the data-collection env of
     * apps/threatsense_runner/collect_and_save.py: EVERY wingman, the agent included, flies the behaviour tree (task
     * :255-266; dc_buffers.actions is ignored), the agent's death does not end the episode (:602-606), compute_observation
     * returns zeros(1) and compute_info (env :112-150) makes every ARMED wingman update its LiDAR and yields its student
     * observation and its last command (the teacher action): dc_buffers.mo_*.  Excludes level5_base_env.
     * 2 = Level52BTEvaluationEnvironment + Level52BTEvaluationTask (level5_eval_2bt_environment.py,
     * .../tasks/level5_2bt_evaluation_task.py; apps/threatsense_runner/evaluation_2bt.py): the same piloting and
     * termination, and in addition no agent is chosen (no draw), no z < -5.99 test, reward 0, no observation at all (no
     * stack kernel, dc_buffers.mo_* unused); kills_per_drone = info agent_kills (slot 0) / allies_kills (slot 1). */
    int32_t level5_multi_obs;
    /* ABI v7, family DC_FAMILY_STAGE03 only: wingmen flown by policies INSIDE the task.
     * lw_driver[j] (j < n_lw, at most 8 wingmen) says who flies wingman j, see DC_DRIVER_*; all zero = the classic tasks.
     *   Exp05_vFinal_Task (exp05_vFinal_task.py:252-260): lw_driver = {DC_DRIVER_LEGACY, DC_DRIVER_NN_ALLY}
     *   Evaluation_Task (evaluation_task.py:89-110,257-277,630-643): one of NN / BT / STOP per configuration["drivers"][j]
     * With any NN / NN_ALLY driver the step has two phases: dc_lw_observe (what compute_lw_observation hands to the
     * policies: dc_buffers.lw_lidar / lw_inertial / lw_present), the caller's policies fill dc_buffers.lw_actions, dc_step.
     * eval_task != 0 = Evaluation_Task + EvaluationEnvironment (evaluation_environment.py:49-130): reward 0, no
     * process_invaders_in_origin, no agent-dead / altitude termination, the step limit only with time_is_limited
     * (TIME_IS_LIMITED), dc_buffers.actions ignored, obs_last_action zero, info rows per wingman in dc_buffers.lw_info. */
    int32_t lw_driver[8];
    int32_t eval_task;
    int32_t time_is_limited;
} dc_config;

/* Caller-owned DEVICE buffers (torch-allocated).  obs_lidar carries state: the reference's
 * FusedLIDAR keeps its last sphere when it cannot update (fused_lidar.py:160-166), so the
 * library leaves an env's slab untouched in that case -- do not scribble on it between steps. */
typedef struct dc_buffers {
    const float* actions;       /* [E,4]  Box([-1,-1,-1,0],[1,1,1,1])  exp02_vFinal_environment.py:197-204 */
    float* obs_lidar;           /* [E,C,13,26]  C = 3 fused / 2 classic */
    float* obs_inertial;        /* [E,15] pos/20, body vel/2.78, euler/pi, body rate/2pi, gun_state[3] */
    float* obs_last_action;     /* [E,4] */
    float* reward;              /* [E] */
    uint8_t* done;              /* [E] terminated (truncated is always False in the reference) */
    int32_t* info;              /* [E,DC_INFO_WORDS] */
    int32_t* lidar_ids;         /* optional [E,13,26]: winning entity slot per cell or -1 */
    float* term_inertial;       /* optional [E,15]: terminal observation of envs that auto-reset */
    float* term_last_action;    /* optional [E,4] */
    double* stats;              /* optional [8]: episodes, sum return, sum length, sum agent_kills,
                                   sum allies_kills, sum deads, sum waves, env steps (atomics) */
    uint8_t* obs_mask;          /* level5 only, mandatory there: [E,DC_LIDAR_STACK] validity mask; obs_lidar is then the
                                   stacked observation [E,DC_LIDAR_STACK,3,13,26] (level5_c1_fusion_environment.py:47-57) */
    int32_t* lidar_hits;        /* optional.  level4/3/2 families: [E,D,2], per entity slot (cell, float bits of r_n) of the
                                   hit it holds in the agent's current sphere, cell = -1 otherwise.  level5: [E,5*D+1,2], the
                                   hit list of the stacked observation, (code, float bits of r_n) with code = sphere*338+cell |
                                   wingman << 11 | age << 12 (age 0 = the observer's own sphere), terminated by code = -1.
                                   Either way a complete sparse description of obs_lidar (dc_host_scatter_sphere /
                                   dc_host_scatter_stack); like obs_lidar it carries state between steps. */
    /* level5 with level5_base_env only, optional (ABI v5): info["student_observation"] of Level5Environment.compute_info
     * (level5_envrionment.py:291-292,342-346) -- the env's SECOND compute_observation call of the step / reset: the same
     * ring, its own fusion draws (FUSE stream, obs_call + 1), every wingman a candidate publisher.  Its inertial_data
     * and last_action equal the returned observation's; info["teacher_observation"] is (zeros(2,13,26), inertial_data,
     * last_action) and needs no buffer.  One more stack_kernel launch per step when bound. */
    float* student_lidar;       /* [E,DC_LIDAR_STACK,3,13,26]; carries state like obs_lidar */
    uint8_t* student_mask;      /* [E,DC_LIDAR_STACK] */
    int32_t* student_hits;      /* optional [E,5*D+1,2]: hit list of student_lidar, same code as the level5 lidar_hits */
    /* level5 with level5_multi_obs only, mandatory there except mo_hits (ABI v6): info["student_observations"] and
     * info["teacher_actions"] of Level5DumbMultiObs.compute_info (level5_dumb_multiobs.py:112-150), one row per wingman
     * slot; rows of wingmen that are not armed (mo_present = 0) are not part of the reference's lists: their stack is
     * emptied, their inertial vector and last command keep the last values. */
    float* mo_lidar;            /* [E,n_lw,DC_LIDAR_STACK,3,13,26]; carries state like obs_lidar */
    uint8_t* mo_mask;           /* [E,n_lw,DC_LIDAR_STACK] */
    float* mo_inertial;         /* [E,n_lw,15] */
    float* mo_last_action;      /* [E,n_lw,4] Quadcopter.last_action (quadcopter.py:415-419); carries state (survives resets) */
    uint8_t* mo_present;        /* [E,n_lw] the wingman is in get_armed_pursuers() at compute_info time */
    int32_t* mo_hits;           /* optional [E,n_lw,5*D+1,2]: hit lists of mo_lidar, level5 code */
    /* policy-driven wingmen (dc_config.lw_driver has an NN / NN_ALLY entry), mandatory then (ABI v7).  Rows of wingmen
     * with another driver are never touched. */
    const float* lw_actions;    /* [E,n_lw,4]  in: the policies' actions (float32, as predict() returns them) for dc_step */
    float* lw_lidar;            /* [E,n_lw,3,13,26]  out of dc_lw_observe: pursuer.lidar sphere; carries state like obs_lidar */
    float* lw_inertial;         /* [E,n_lw,15] out of dc_lw_observe: inertial + gun vector of every ARMED policy-driven wingman */
    uint8_t* lw_present;        /* [E,n_lw]    out of dc_lw_observe: the wingman is served by its policy in the coming step */
    int32_t* lw_info;           /* optional [E,n_lw,4] out of dc_step: lw_kills, armed, lw_munitions, 0 at compute_info time */
} dc_buffers;

typedef struct dc_sim dc_sim;

int dc_create(const dc_config* cfg, int device, dc_sim** out);
int dc_bind(dc_sim* sim, const dc_buffers* buffers);
/* mask: optional device pointer [E] (non-zero = reset this env); NULL resets every env. */
int dc_reset(dc_sim* sim, const uint8_t* mask, void* stream);
int dc_step(dc_sim* sim, void* stream);
/* First phase of a step when wingmen are flown by policies inside the task (dc_config.lw_driver): the observation
 * Evaluation_Task.compute_lw_observation (evaluation_task.py:283-312) / Exp05_vFinal_Task.compute_lw_observation
 * (exp05_vFinal_task.py:265-296) builds at on_step_start for every policy-driven wingman -> dc_buffers.lw_lidar,
 * lw_inertial, lw_present.  ("last_action" of that observation is the task's shared variable: the action of whichever
 * policy-driven wingman was served last, zero after a reset -- host state, see dronechase_b200.drivers.)  Call it once
 * before every dc_step, also before the first step after dc_reset. */
int dc_lw_observe(dc_sim* sim, void* stream);
/* Point the next dc_step at another [E,4] float device buffer (16-byte aligned) without re-binding
 * everything: the zero-copy path for a policy whose action tensor changes address every step. */
int dc_set_actions(dc_sim* sim, const float* actions);
/* dc_step may be captured into a CUDA graph (it only enqueues kernels and events).  The library ping-pongs internal
 * buffers by a step parity that is a kernel argument, so capture TWO consecutive dc_step calls into two graphs and replay
 * them alternately; after every replay call dc_note_graph_replay so that the host-side parity (used by dc_reset and
 * dc_copy_state) follows the device.  dronechase_b200.sim.BatchedThreatEngageEnv.step_graph does exactly this. */
int dc_note_graph_replay(dc_sim* sim);
void dc_destroy(dc_sim* sim);
const char* dc_last_error(void);

/* Parity harness: copy the raw state to/from HOST memory (synchronises).
 *   which = 0: drone state, element type float (F32) or double (F64), layout [DC_STATE_QUADS][E*D][4]
 *              quad 0 pos.xyz|flag word (bit0 armed, bit1 in-offsets-snapshot, bits2-3 nav state, bits 8.. ammo)
 *                   1 quat xyzw   2 vel(world).xyz|0   3 omega(body).xyz|0
 *                   4 motor throttle[4]   5-10 PID words (oracle/dynamics.py PID_SLOTS)
 *                   11 imu_pos.xyz|last_fired_step      12 formation.xyz|0
 *   which = 1: env scalars, int32 [E][DC_ENV_WORDS]: step, max_step, round, agent_kills, allies_kills,
 *              deads, building_life, hit_ctr, spawn_ctr, phys_ctr, last_closest (double, 2 words),
 *              episode_return (float), episode_steps, initialised, spare
 *   which = 2: fixed LW spawn points, double [E][n_lw][3]
 * to_device != 0 writes the host buffer into the sim. */
int dc_copy_state(dc_sim* sim, int which, void* host, size_t bytes, int to_device);
size_t dc_state_bytes(const dc_sim* sim, int which);

/* Stand-alone projection LiDAR (threatsense microbenchmark, BASELINE config 4):
 * n_obs observers per env see the env's n_ent entities; observer o of env e is entity obs_slot[o].
 *   pos [E,n_ent,3] f32, quat [E,n_ent,4] f32 xyzw, type [n_ent] int32 (EntityType value),
 *   alive [E,n_ent] u8, sphere out [E,n_obs,C,13,26] f32, ids out (optional) [E,n_obs,13,26] i32. */
int dc_lidar_project(const float* pos, const float* quat, const int32_t* type, const uint8_t* alive,
                     const int32_t* obs_slot, int32_t n_envs, int32_t n_ent, int32_t n_obs,
                     int32_t flavour, double radius, float* sphere, int32_t* ids, void* stream);

/* Opt-in ray-cast variant of the sensor (not in the reference, which only projects centres): one ray per
 * cell centre against every entity's bounding sphere (radius [n_ent] f32, metres), nearest hit wins, and every
 * entity also claims the cell of its centre at its centre distance -- with radii -> 0 the result equals
 * dc_lidar_project(flavour = DC_LIDAR_FUSED).  Same tensors as dc_lidar_project, 3 channels. */
int dc_lidar_raycast(const float* pos, const float* quat, const float* radius_per_entity, const int32_t* type,
                     const uint8_t* alive, const int32_t* obs_slot, int32_t n_envs, int32_t n_ent, int32_t n_obs,
                     double max_range, float* sphere, int32_t* ids, void* stream);

/* HOST helper for adapters that hand numpy arrays to the reference's training code (SB3 VecEnv contract): rebuilds the
 * dense sphere observation in host memory from the sparse hit list instead of moving 4 KB per env over PCIe.
 *   dense [E,C,13,26] f32 host array that currently shows prev_hits (all ones when prev_hits is all -1);
 *   prev_hits / hits: host copies of dc_buffers.lidar_hits ([E,D,2] int32) for the step dense shows / the new step.
 * The cells of prev_hits go back to 1.0, then hits are written: r_n, EntityType/5 (0.6 wingman slots < n_lw, 0.2
 * munitions), and 0.1 in the third channel when C == 3 -- what FusedLIDAR.update_data / LIDAR.update_data leave in the
 * sphere (fused_lidar.py:143-217, lidar.py:263-280).  Runs on n_threads host threads; touches no device. */
int dc_host_scatter_sphere(float* dense, const int32_t* prev_hits, const int32_t* hits, int32_t n_envs, int32_t n_drones,
                           int32_t n_lw, int32_t channels, int32_t n_threads);

/* Same for the level5 stacked observation: dense [E,6,3,13,26], prev_hits / hits host copies of the level5 lidar_hits
 * ([E,5*n_drones+1,2]); flag = 0.6 / 0.2, time = 0.1 for the observer's own sphere, age/10 for a neighbour snapshot
 * (fused_lidar.py:223-326, lidar_math.py:262-311). */
int dc_host_scatter_stack(float* dense, const int32_t* prev_hits, const int32_t* hits, int32_t n_envs, int32_t n_drones,
                          int32_t n_threads);

/* Number of kernel launches this library has enqueued so far in this process. */
/* Device-side twin of dc_host_scatter_sphere: dense[r] (channels,13,26) = empty sphere + the hits of row
 * (row_index ? row_index[r] : r) of `hits` ([rows, n_drones, 2] int32, the layout of dc_buffers.lidar_hits for the
 * level4/3/2 families).  Lets a rollout keep its LiDAR observations as hit lists (56 B instead of 4 KB per env step for
 * 7 drones) and rebuild minibatches on demand: the device-resident replacement of the SB3 rollout buffer's numpy/PCIe
 * round trip (src/core/rl_framework/utils/pipeline.py:214-241).  All pointers are device pointers. */
int dc_scatter_hits(const int32_t* hits, const int64_t* row_index, int64_t n_rows, int32_t n_drones, int32_t n_lw,
                    int32_t channels, float* dense, void* stream);

/* The same for the level5 stacked observation (device-side twin of dc_host_scatter_stack): dense[r] (6,3,13,26) = six
 * empty spheres + the hit list of row (row_index ? row_index[r] : r) of `hits` ([rows, 5*n_drones+1, 2] int32, the level5
 * layout of dc_buffers.lidar_hits / student_hits).  24 KB per env step shrink to the list (at most 8 * (5 D + 1) bytes);
 * the validity mask (6 bytes) is stored beside it by the caller.  dense must be 16-byte aligned. */
int dc_scatter_stack(const int32_t* hits, const int64_t* row_index, int64_t n_rows, int32_t n_drones, float* dense,
                     void* stream);

/* Zero-copy observation for the numpy-facing adapter (SB3 VecEnv contract: dense (C,13,26) arrays in HOST memory).
 * dc_host_register page-locks a host range and maps it into the device address space (cudaHostRegister Mapped|Portable);
 * *device_ptr is the address kernels may use for it.  dc_mirror_hits then keeps such an array equal to the sphere
 * observation with a few 4-byte PCIe writes per env and step: `shown_hits` (device, [E,D,2] int32, in/out) holds the hits
 * the array currently shows (all -1 for an all-ones array) and is brought to `hits` (dc_buffers.lidar_hits).  The values
 * written are those of dc_host_scatter_sphere; after the stream is synchronised the host array equals obs_lidar bit for
 * bit.  Level4/3/2 families only (the level5 stack changes most of its cells every step: use dc_host_scatter_stack). */
int dc_host_register(void* host, size_t bytes, void** device_ptr);
int dc_host_unregister(void* host);
int dc_mirror_hits(int32_t* shown_hits, const int32_t* hits, int32_t n_envs, int32_t n_drones, int32_t n_lw, int32_t channels,
                   float* dense, void* stream);

/* The third way to keep a dense host array equal to the sphere: the update of dc_mirror_hits as a LIST.  `out_pairs`
 * (device, 8-byte aligned, 2 * (1 + 6 * n_envs * n_drones) int32 in the worst case) receives the number of pairs in
 * out_pairs[0] and, from out_pairs[2] on, (flat float index into dense [E, C, 13, 26], float bits) pairs that bring an array
 * showing `shown_hits` to `hits`; `shown_hits` is updated.  The pairs of one call never repeat an index (an un-write whose
 * cell another slot enters in the same step is dropped), so the host may store them in any order with any number of
 * threads: copy out_pairs[0..] to pinned memory and hand it to dc_host_apply_pairs.  A list of the changed words crosses
 * PCIe on the copy engines in tens of microseconds; the posted 4-byte writes of dc_mirror_hits take 0.4 ms per 65,536 envs. */
int dc_diff_hits(int32_t* shown_hits, const int32_t* hits, int32_t n_envs, int32_t n_drones, int32_t n_lw, int32_t channels,
                 int32_t* out_pairs, void* stream);
/* dense[index] = value for n_pairs (index, float bits) pairs in host memory (pairs points at the first PAIR, not at the
 * count), on n_threads host threads.  Needs no device. */
int dc_host_apply_pairs(float* dense, const int32_t* pairs, int64_t n_pairs, int32_t n_threads);

uint64_t dc_launch_count(void);

/* Binding self-check for hosts that mirror the structs by hand (ctypes, cgo, JNI): which = 0 -> DC_ABI_VERSION,
 * 1 -> sizeof(dc_config), 2 -> sizeof(dc_buffers); anything else -> 0.  Needs no device. */
size_t dc_abi_info(int which);

/* 1 when `quad` (DC_QUAD_PARAM_WORDS doubles, the layout of dc_config.quad) is the built-in cf2x model -- every word but the
 * motor noise ratio [8] and the ground height [15], which stay run-time values -- so that the float32 dynamics run the
 * instantiation with the model folded into the code; 0 otherwise (same results to float32 rounding, run-time constants).
 * Mirrors dronechase_b200/config.py CF2X (the reference's drone: PyFlyt cf2x.yaml behind quadcopter.py:143-152).  Needs no device. */
int dc_quad_is_builtin(const double* quad);

/* ---- The agent's policy on the device (SURVEY.md 8(f) rank 1): model.predict(obs, deterministic=True) of the reference's SB3
 * PPO -- LidarInertialActionExtractor (src/core/rl_framework/agents/policies/ppo_policies.py:234-342: Conv2d(C,32,k4,s4)-ReLU-
 * Conv2d(32,64,k2,s2)-ReLU-Flatten over the sphere, 3 x 128 MLPs over inertial_data and last_action, Linear(448,
 * features_dim)-ReLU), mlp_extractor.policy_net (net_arch["pi"], ppo_policies.py:150-156), action_net, clip to the action
 * box -- as ONE kernel launch that reads the observation tensors of dc_buffers where they are and writes the action tensor
 * dc_step consumes.  Replaces, on the rollout path, the observation round trip of src/core/rl_framework/utils/pipeline.py:214-241
 * (SubprocVecEnv -> numpy -> torch policy -> numpy -> pipes).
 * All weight pointers are DEVICE (or device-accessible) pointers in torch layout: Linear [out][in] row-major, Conv2d
 * [out][in][kh][kw]; they are read once by dc_policy_create (re-laid out for the tensor cores) and need not outlive it. */
typedef struct dc_policy dc_policy;
typedef struct dc_policy_weights {
    int32_t lidar_channels;       /* C of the (C,13,26) sphere: 1..3 */
    int32_t features_dim;         /* 64, 128, 192 or 256 */
    int32_t n_pi;                 /* hidden layers of pi: 0..8 */
    int32_t pi[8];                /* their widths: multiples of 64, <= 256; the last one <= 1024 */
    int32_t activation;           /* of the pi layers: 1 = ReLU, 2 = Tanh (SB3's default) */
    const float* conv1_w; const float* conv1_b;      /* [32][C][4][4], [32] */
    const float* conv2_w; const float* conv2_b;      /* [64][32][2][2], [64] */
    const float* inertial_w[3]; const float* inertial_b[3];   /* [128][15], [128][128], [128][128] */
    const float* action_w[3]; const float* action_b[3];       /* [128][4], [128][128], [128][128] */
    const float* final_w; const float* final_b;      /* [features_dim][448] over (lidar 192 | inertial 128 | action 128) */
    const float* pi_w[8]; const float* pi_b[8];
    const float* head_w; const float* head_b;        /* action_net: [4][last width], [4] */
    float low[4], high[4];                           /* the action box the mean action is clipped to */
} dc_policy_weights;
int dc_policy_create(const dc_policy_weights* weights, int device, dc_policy** out);
/* actions[e] = clip(action_net(pi(features(lidar[e], inertial[e], last_action[e])))) for n_envs rows; lidar [n_envs][C][13][26],
 * inertial [n_envs][15], last_action [n_envs][4], actions [n_envs][4], float32 device pointers.  precision 0: every product as
 * three TF32 MMAs (head/tail split, float32-grade: within 2e-5 of a float32 evaluation); 1: plain TF32 operands, float32
 * accumulate (within 5e-3).  Stream-ordered on `stream`; the same bits on every run. */
int dc_policy_forward(dc_policy* policy, const float* lidar, const float* inertial, const float* last_action, int64_t n_envs,
                      float* actions, int32_t precision, void* stream);
void dc_policy_destroy(dc_policy* policy);

/* ---- PPO rollout collection on the device: what SB3's OnPolicyAlgorithm.collect_rollouts asks of the policy each step (a sampled
 * action, its log-probability, V(s)) and, after the last step, RolloutBuffer.compute_returns_and_advantage.
 * dc_value_weights: the rest of SB3's ActorCriticPolicy with a shared features extractor and net_arch = dict(pi=..., vf=...):
 * mlp_extractor.value_net (hidden layers over the features, the activation of pi), value_net, and the DiagGaussian's log_std.
 * Device pointers in torch layout, read once by dc_policy_create_ac. */
typedef struct dc_value_weights {
    int32_t n_vf; int32_t vf[8];                 /* hidden widths of mlp_extractor.value_net: 0..8 layers, the rules of pi */
    const float* vf_w[8]; const float* vf_b[8];
    const float* value_w; const float* value_b;  /* value_net: [1][last width], [1] */
    const float* log_std;                        /* [4], read once, like the weights */
} dc_value_weights;
/* A policy that dc_policy_act can run as well as dc_policy_forward (which runs the plain kernel on it, unchanged). */
int dc_policy_create_ac(const dc_policy_weights* weights, const dc_value_weights* value, int device, dc_policy** out);
/* One launch for n_envs rows.  mean = action_net(...) (unclipped), value[e] = V(s).  sample = 1: eps = four standard normals
 * (Box-Muller on the Philox4x32-10 block of key seed, counter (counter, 5, env_offset + e, 0)), raw_actions[e] = mean +
 * exp(log_std) * eps, env_actions[e] = clip(raw) to the action box, log_prob[e] = sum_k(-eps_k^2 / 2 - log_std_k) - 2 log(2 pi).
 * sample = 0: env_actions = clip(mean), bit for bit what dc_policy_forward writes; raw_actions and log_prob are not written and
 * may be NULL.  The same bits on every run and for any split of the rows (pass the split's env_offset). */
int dc_policy_act(dc_policy* policy, const float* lidar, const float* inertial, const float* last_action, int64_t n_envs,
                  uint64_t seed, int64_t env_offset, uint32_t counter, int32_t sample,
                  float* env_actions /*[n][4] clipped*/, float* raw_actions /*[n][4], NULL if !sample*/,
                  float* log_prob /*[n], NULL if !sample*/, float* value /*[n]*/, int32_t precision, void* stream);
/* Generalized advantage estimation over a [T][E] rollout, float32 device arrays (dones uint8: 1 = the episode ended AFTER step
 * t): delta_t = r_t + gamma V_{t+1} (1 - d_t) - V_t with V_T = last_values [E]; A_t = delta_t + gamma lambda (1 - d_t) A_{t+1};
 * returns = A + V.  SB3's compute_returns_and_advantage with episode_starts[t + 1] = dones[t]. */
int dc_gae(const float* rewards, const uint8_t* dones, const float* values, const float* last_values, int64_t T, int64_t E,
           float gamma, float gae_lambda, float* advantages, float* returns, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DRONECHASE_B200_H */

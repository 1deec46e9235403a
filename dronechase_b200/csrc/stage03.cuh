// dronechase_b200 -- the stage03 env step as two kernels per step.
//
//   dyn_kernel   one thread per ARMED drone, taken from a device-resident work list:
//                scripted pilot / RL action -> setpoint   Task.on_step_start  exp02_vFinal_task.py:231-242,275-282
//                16 physics substeps in registers          advance_step        exp02_vFinal_environment.py:179-188
//   env_kernel   every WARP owns `epw` consecutive envs and their drone slots through all phases (no block barrier):
//                P0  slot pass: flag words, fresh IMU positions, remembered sphere hits into shared memory
//                P3  env pass (one lane per env): engagement / reward / termination / info / obs vector /
//                    waves / auto-reset          Task.on_step_middle :284-318, Task.on_step_end :320-332
//                    spawn pass: the munition waves P3 asked for, one lane per munition
//                P5  slot pass: events -> state, next step's work list (warp-level compaction)
//                P4  projection LiDAR + incremental sphere  compute_observation exp02_vFinal_environment.py:206-234
// Only armed drones are simulated (the reference drops disarmed ones from active_drones,
// entities_manager.py:230-232).  The work list is rebuilt by env_kernel from the final armed flags, so
// every lane of every dynamics warp carries a live drone whatever the wave, and the two kernels can
// each run at their own register budget / occupancy.
#pragma once
#include "../../include/dronechase_b200.h"
#include "common.cuh"
#include "lidar.cuh"
#include "quad_dynamics.cuh"

namespace dc {

// The task families both step kernels are compiled for, their template parameter FAM: every family gets its own
// specialisation without the other families' branches (each runtime family switch had cost ~6 % of the step).  The first
// four are dc_config.family.  FAM_L5_MULTI (dc_config.level5_multi_obs: Level5DumbMultiObs, Level52BTEvaluationEnvironment)
// is split from FAM_L5 so that its extra code costs the hot level5 kernels nothing (it did: + 2.8 % on level5_c1 as
// run-time branches); FAM_DRIVEN is stage03 with wingmen flown by policies inside the task (driven.cuh).
enum { FAM_STAGE03 = DC_FAMILY_STAGE03, FAM_STAGE02 = DC_FAMILY_STAGE02, FAM_STAGE01 = DC_FAMILY_STAGE01,
       FAM_L5 = DC_FAMILY_LEVEL5, FAM_L5_MULTI = 4, FAM_DRIVEN = 5, FAM_RAYCAST = 6 };
// FAM_RAYCAST names an env_kernel instantiation only: the stage03 step of a sim whose agent senses with the ray-cast LiDAR
// (dc_config.lidar = DC_LIDAR_RAYCAST), which also exports what its LiDAR pass projected from (raycast_env.cuh).
// the level5 (threatsense) envs: the RL agent is a random wingman, every wingman keeps an IMU record and a LiDAR ring
__host__ __device__ constexpr bool fam_l5(int f) { return f == FAM_L5 || f == FAM_L5_MULTI; }
// the families whose munitions come in waves, spawned by env_kernel's spawn pass
__host__ __device__ constexpr bool fam_waves(int f) { return f == FAM_STAGE03 || f == FAM_DRIVEN || fam_l5(f); }

#ifndef DC_DYN_THREADS
#define DC_DYN_THREADS 128
#endif
constexpr int DYN_THREADS = DC_DYN_THREADS;
constexpr int ENV_THREADS = 128;
#ifndef DC_ENV_MIN_BLOCKS
#define DC_ENV_MIN_BLOCKS 4
#endif
#ifndef DC_DYN_MIN_BLOCKS
#define DC_DYN_MIN_BLOCKS 6
#endif
enum { MODE_STEP = 0, MODE_RESET = 1 };
// dc_config.lw_driver: who flies a wingman.  LEGACY = the task's own rule (slot 0 = dc_buffers.actions, the others
// TaskParams::ally_mode); NN = dc_buffers.lw_actions whenever armed; BT = LoyalWingmanBehaviorTree whenever armed; STOP =
// drive([0,0,0,1]) (zero velocity); NN_ALLY = lw_actions, but only behind an armed pursuer (exp05: get_armed_pursuers()[1:])
enum { DRV_LEGACY = 0, DRV_NN = 1, DRV_BT = 2, DRV_STOP = 3, DRV_NN_ALLY = 4 };
enum { NAV_WAIT = 0, NAV_WINGMAN = 1, NAV_BUILDING = 2 };
// flag word per drone slot: bit0 armed, bit1 member of the offsets snapshot, bits 8.. ammunition
enum { F_ARMED = 1, F_OFF = 2, F_SNAP = 4, F_PENDING = 16, F_PENDING2 = 32, F_AMMO_SHIFT = 8 };   // F_PENDING*: stage01 extra updates owed (see dyn_kernel)
// F_SNAP: the drone has a readable (slot 1) snapshot in the LiDAR rings -- it was armed at the last AGENT_STEP_BROADCAST and
// has not been disarmed (MessageHub.terminate) or re-armed (slot 0 only, STABLE_DELTA_STEP = 1) since; what a policy-driven
// wingman's update_lidar sees at the NEXT on_step_start (lw_obs_kernel)
// per-drone event word built by the env pass
enum { EV_LIVE = 1, EV_OFF = 2, EV_MID = 4, EV_ZEROED = 8, EV_REPLACED = 16, EV_REARMED = 32, EV_WAS_ARMED = 64, EV_PENDING = 128, EV_PENDING2 = 256, EV_LWIN = 512, EV_SPAWNJOB = 1024, EV_SNAP = 2048 };
// env scalar words
enum { W_STEP = 0, W_MAX_STEP, W_ROUND, W_AGENT_KILLS, W_ALLIES_KILLS, W_DEADS, W_BUILDING, W_HIT_CTR,
       W_SPAWN_CTR, W_PHYS_CTR, W_LAST_CLOSEST_LO, W_LAST_CLOSEST_HI, W_EP_RETURN, W_EP_STEPS, W_INIT, W_SPARE };
// envflag bits
enum { EF_LIDAR = 1, EF_NAV_RESET = 2, EF_FIRST = 8 };
// per-env agent imu record (global, AG_WORDS scalars per env)
// level5 per-env words (SimPtrs::env5)
enum { W5_AGENT = 0, W5_GUN_STEP, W5_REGISTERED, W5_OBS_CALL, W5_LAST_DIST_LO, W5_LAST_DIST_HI, W5_STACK_MODE, W5_PREV_N, ENV5_WORDS = 8 };
enum { STACK_KEEP = 0, STACK_BUILD = 1, STACK_EMPTY = 2 };
constexpr int N_STACK = 6;       // n_neighbors_max + 1 (fused_lidar.py:59,307)
constexpr int RING = 10;         // LiDARBufferManager max_buffer_size (base_lidar.py:37)
enum { AG_UB = 0, AG_VB, AG_WB, AG_ROLL, AG_PITCH, AG_YAW, AG_P, AG_Q, AG_R, AG_QX, AG_QY, AG_QZ, AG_QW, AG_WORDS = 16 };

struct TaskParams {
    int n_envs, n_lw, n_lm, D;
    int munition, step_increment, max_step, initial_round, substeps;
    int lm_nav, ally_mode, reward, lidar, fixed_lw_spawn, auto_reset;
    int family;              // 0 stage03 (level4 tasks), 1 stage02 (level3 L3Stage1), 2 stage01 (level2 modified_v2),
                             // 3 level5 (threatsense Level5C1FusionTask)
    int initial_invaders, invaders_per_round, max_rounds;   // level5 waves (level5_c1_fusion_task.py:83-90)
    int n_rec;               // imu records per env: 1 (the agent, slot 0) or n_lw (level5: every wingman)
    int l5_base;             // level5: base Level5Environment observation protocol (dc_config.level5_base_env)
    int l5_multi;            // level5: Level5DumbMultiObs protocol (dc_config.level5_multi_obs): every wingman flies the
                             // behaviour tree, every ARMED wingman observes, the agent's death does not end the episode
    int l5_eval;             // level5: Level52BTEvaluationEnvironment (dc_config.level5_multi_obs == 2): l5_multi's piloting
                             // and termination, plus no agent draw, no z test, no reward, no observation
    int support_munition;    // stage02: Gun() default of the support wingman
    // FAM_DRIVEN: wingmen flown by policies INSIDE the task -- Evaluation_Task
    // (evaluation_task.py:257-277,630-643) and Exp05_vFinal_Task (exp05_vFinal_task.py:252-260)
    int lw_driver[8];        // per wingman slot: DRV_*
    int eval_task;           // Evaluation_Task: no reward, no origin processing, no agent-dead / altitude termination,
                             // per-wingman kill counters, env last_action always zero
    int time_limited;        // Evaluation_Task TIME_IS_LIMITED: the step limit only ends the episode when set
    double respawn_r0, respawn_r1;   // stage02: disarmed munitions reappear on r in U(r0, r1)
    uint32_t env_offset, k0, k1;
    double dome, born, lw_spawn, expl, shoot, cooldown, fire_p, lm_speed, bt_speed, ally_stop, vel_bonus;
    double building[3];
    double acos_born, acos_lw;   // acos(min(4, r) / r) for r = born and r = lw_spawn (generate_positions' lower phi bound)
};

// Device state of one sim.  Quads are [quad][E*D]: 0 pos, 1 quat, 2 vel, 3 omega, 4 throttle, 5-9 PID
// (mode 6), 10 PID (mode 7), 11 unused, 12 formation.  imu[2] is ping-pong: imu[p] = last step's IMU
// position | last_fired_step (the offsets snapshot), imu[1-p] = this step's.
template <typename R> struct SimPtrs {
    V4<R>* state;
    V4<R>* imu[2];
    int32_t* flagw;          // [E*D]
    unsigned char* nav;      // [E*D]
    R* agent;                // [E][AG_WORDS]
    int32_t* env;            // [E][ENV_WORDS]
    double* lw_init;         // [E][n_lw][3]
    int32_t* items[2];       // work lists (armed slots), ping-pong like imu
    int32_t* count;          // [2]
    double* last_dist;       // [E][n_lm] stage02: previous step's agent->munition distances (OffsetHandler.last_offsets)
    int2* sphere_desc;       // [E*D] (cell, float bits of r_n) of the entity that holds a cell of the agent's
                             // current sphere, cell = -1 otherwise: lets a kept sphere be re-materialised
    // ---- level5 (threatsense) only: the agent's LiDAR ring restricted to what read_data can reach ----
    int32_t* env5;           // [E][ENV5_WORDS]
    float* ring_pose;        // [E][n_lw][RING][8]  float32 snapshot pose (pos xyz, quat xyzw, pad) of wingman P at step t
    int32_t* ring_meta;      // [E][n_lw][RING][D]  kept feature of P about entity d at step t: cell | type << 16, or -1
    double* ring_feat;       // [E][n_lw][RING][D][3]  (r_n, theta, phi) float64 as FusedLIDAR.features keeps them
    int2* stack_prev;        // [E][5*D+1]  hit list of the stacked observation (level5_stack.cuh), -1 terminated
    int32_t* mo_prev_n;      // marked cells of the student stack [E] / of the multi-observer stacks [E][n_lw]
                             // (the agent's own count is the env5 word W5_PREV_N: 32-byte rows)
    // ---- FAM_DRIVEN only ----
    int2* lw_desc;           // [E][n_lw][D]  like sphere_desc, for the per-wingman spheres dc_buffers.lw_lidar
    int32_t* lw_kills;       // [E][n_lw]     Evaluation_Task.lw_kills (successful shots of the episode)
};

template <typename R> struct StepArgs {
    TaskParams t;
    QuadParams<R> q;
    SimPtrs<R> p;
    int parity;              // imu[parity] / items[parity] are the inputs of this step
    const float* actions;
    float* obs_lidar; float* obs_inertial; float* obs_last_action;
    float* reward; uint8_t* done; int32_t* info; int32_t* lidar_ids;
    float* term_inertial; float* term_last_action; double* stats;
    uint8_t* obs_mask;       // level5: [E][N_STACK] validity mask of the stacked spheres
    // level5 multi-observer (Level5DumbMultiObs.compute_info): per wingman
    float* mo_inertial;      // [E][n_lw][15]
    float* mo_last_action;   // [E][n_lw][4]  the wingman's last command = info["teacher_actions"]
    uint8_t* mo_present;     // [E][n_lw]     armed at compute_info time
    // FAM_DRIVEN (policy-driven wingmen): what compute_lw_observation (evaluation_task.py:283-312) hands to the policies
    const float* lw_actions; // [E][n_lw][4]  actions of the policy-driven wingmen for THIS step
    float* lw_lidar;         // [E][n_lw][C][13][26]  sphere of every policy-driven wingman as of the NEXT on_step_start
    float* lw_inertial;      // [E][n_lw][15]
    uint8_t* lw_present;     // [E][n_lw]     the wingman will be served by its policy at the next on_step_start
    int32_t* lw_info;        // [E][n_lw][4]  compute_info rows: lw_kills, armed, munition, 0
    const uint8_t* reset_mask;
    int epb;                 // envs per block of env_kernel
    int epw;                 // envs per warp of env_kernel (<= 32)
    uint32_t div_m;          // slot / D == (slot * div_m) >> 20 for every slot index of a block (checked by dc_create)
    __device__ int env_of(int s) const { return (int)(((uint32_t)s * div_m) >> 20); }     // block slot -> block env
    int tl_slot;             // profiling builds (DC_PROFILE_PHASES): row of g_tl this launch stamps
    alignas(16) uint32_t rk[20];   // Philox round keys of (t.k0, t.k1) for philox4x32_10_rk (dyn_kernel's motor noise)
    float4* ray_snap;        // env_kernel<FAM_RAYCAST>: [E*D] export of P4's inputs (RS_*); last, so no other field moves
};

#ifdef DC_PROFILE_PHASES      // launch timeline: first block start / last warp end of every step kernel, in globaltimer ns
__device__ unsigned long long g_tl[256][2];
__device__ __forceinline__ unsigned long long gtime() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
#define DC_TL_BEGIN(slot) do { if ((threadIdx.x & 31) == 0) atomicMin(&g_tl[(slot) & 255][0], gtime()); } while (0)
#define DC_TL_END(slot) do { if ((threadIdx.x & 31) == 0) atomicMax(&g_tl[(slot) & 255][1], gtime()); } while (0)
#else
#define DC_TL_BEGIN(slot) do { } while (0)
#define DC_TL_END(slot) do { } while (0)
#endif

__device__ __forceinline__ double norm3(double x, double y, double z) { return sqrt(x * x + y * y + z * z); }
__device__ __forceinline__ double sq3(double x, double y, double z) { return x * x + y * y + z * z; }

// ================================================================================================
// dyn_kernel
// ================================================================================================
// The state words a drone carries through dyn_kernel's substeps, listed once in move(): quads 0-4 (position, quaternion,
// velocity, body rate, throttle), then the PID words.  load() and store() are move(); the prefetch skips what move() skips.
template <typename R, int FAM, bool BUILTIN> struct DroneWords {
    static constexpr int NPID = FAM == FAM_STAGE01 ? 6 : 5;                       // quad 10 holds the mode-7 words
    // The folded cf2x model (BUILTIN) has ki = kd = 0 in the angle loop and kd = 0 in the yaw-rate loop: of the 20 mode-6
    // controller words only 11 are ever read -- ang_vel integrators 0..2 and previous errors 3, 4, lin_vel 12..15, z_vel 16, 17.
    // The others are neither loaded nor written back (they keep what the last reset left): 9 registers less across the
    // substep loop and 56 bytes less traffic per drone and direction.
    static constexpr bool PID_DIET = BUILTIN && sizeof(R) == 4 && FAM != FAM_STAGE01;
    __device__ __forceinline__ static void prefetch(const V4<R>* gp, long long stride) {
#pragma unroll
        for (int q = 0; q < 10; ++q)                         // quad 10 is loaded but not prefetched
            if (!(PID_DIET && q == 7)) asm volatile("prefetch.global.L2 [%0];" :: "l"(gp + q * stride));
    }
    // one 16-byte quad (d == nullptr: its fourth word is not carried, stored as 0), or one word on its own
    template <bool ST> __device__ __forceinline__ static void quad(V4<R>* p, R& a, R& b, R& c, R* d) {
        if constexpr (ST) st4(p, V4<R>{a, b, c, d ? *d : (R)0});
        else { const V4<R> v = ld4(p); a = v.x; b = v.y; c = v.z; if (d) *d = v.w; }
    }
    template <bool ST> __device__ __forceinline__ static void word(R* p, R& a) { if constexpr (ST) *p = a; else a = *p; }
    template <bool ST> __device__ __forceinline__ static void move(Drone<R>& st, V4<R>* gp, long long stride) {
        quad<ST>(gp, st.px, st.py, st.pz, nullptr);
        quad<ST>(gp + stride, st.qx, st.qy, st.qz, &st.qw);
        quad<ST>(gp + 2 * stride, st.vx, st.vy, st.vz, nullptr);
        quad<ST>(gp + 3 * stride, st.wx, st.wy, st.wz, nullptr);
        quad<ST>(gp + 4 * stride, st.thr[0], st.thr[1], st.thr[2], &st.thr[3]);
        if constexpr (PID_DIET) {
            if constexpr (!ST)
#pragma unroll
                for (int k = 0; k < 24; ++k) st.pid[k] = 0;
            quad<ST>(gp + 5 * stride, st.pid[0], st.pid[1], st.pid[2], &st.pid[3]);
            word<ST>(reinterpret_cast<R*>(gp + 6 * stride), st.pid[4]);
            quad<ST>(gp + 8 * stride, st.pid[12], st.pid[13], st.pid[14], &st.pid[15]);
            word<ST>(reinterpret_cast<R*>(gp + 9 * stride), st.pid[16]); word<ST>(reinterpret_cast<R*>(gp + 9 * stride) + 1, st.pid[17]);
        } else {
#pragma unroll
            for (int k = 0; k < NPID; ++k) quad<ST>(gp + (5 + k) * stride, st.pid[4 * k], st.pid[4 * k + 1], st.pid[4 * k + 2], &st.pid[4 * k + 3]);
        }
    }
    __device__ __forceinline__ static void load(Drone<R>& st, V4<R>* gp, long long stride) { move<false>(st, gp, stride); }
    __device__ __forceinline__ static void store(Drone<R>& st, V4<R>* gp, long long stride) { move<true>(st, gp, stride); }
};

// FAM: FAM_* above.  BUILTIN (float32 only): the drone model is the built-in cf2x, folded into the code (quad_dynamics.cuh Cf2x).
template <typename R, bool NOISE, int FAM, bool BUILTIN = false>
__global__ void __launch_bounds__(DYN_THREADS, (sizeof(R) == 4 ? DC_DYN_MIN_BLOCKS : 2)) dyn_kernel(const StepArgs<R> A) {
    const TaskParams& T = A.t;
    const int par = A.parity;
    // launched with programmatic stream serialisation: nothing is read or written before the previous grid (the
    // previous step's env_kernel) has completed
    asm volatile("griddepcontrol.wait;" ::: "memory");
    DC_TL_BEGIN(A.tl_slot);
    const int n_items = A.p.count[par];
    if (blockIdx.x == 0 && threadIdx.x == 0) A.p.count[par ^ 1] = 0;      // env_kernel refills it after us
    const int it = blockIdx.x * DYN_THREADS + threadIdx.x;
    if (it >= n_items) { DC_TL_END(A.tl_slot); return; }
    const int D = T.D;
    const int s = A.p.items[par][it];                 // global slot = env * D + d
    const int env = s / D, d = s - env * D;
    const long long b = (long long)env * D;
    const long long stride = (long long)T.n_envs * D;
    const bool is_lw = d < T.n_lw;
    const V4<R>* snap = A.p.imu[par];
    // The pilots below walk a chain of dependent loads (flags -> neighbour snapshots -> formation point) before the drone's
    // own state is touched: ask for the state lines now so that they arrive under that chain (no registers held).
    using Words = DroneWords<R, FAM, BUILTIN>;
    Words::prefetch(A.p.state + s, stride);
    asm volatile("prefetch.global.L2 [%0];" :: "l"(A.p.env + (long long)env * ENV_WORDS));
    const V4<R> own = ld4(snap + s);                  // imu position of the previous step | last_fired
    const double mx = own.x, my = own.y, mz = own.z;

    // ---- scripted pilots / RL action -> mode-6 setpoint -------------------------------------------
    double cmd[4] = {0, 0, 0, 0};
    bool driven = false;
    // level5: the RL agent is a random wingman (entities_manager.py:350-383) and guns/tasks read the step of the
    // last AGENT_STEP_BROADCAST, which the id clash with munition 0 can zero (see env_kernel)
    const int agent_slot = fam_l5(FAM) ? A.p.env5[(long long)env * ENV5_WORDS + W5_AGENT] : 0;
    // behaviour tree (LoyalWingmanBehaviorTree, loyalwingman_navigator.py:79-86): gun available (or empty) -> chase, else formation
    auto bt_command = [&]() {
        const int ammo = A.p.flagw[s] >> F_AMMO_SHIFT;
        const int cur_step = fam_l5(FAM) ? A.p.env5[(long long)env * ENV5_WORDS + W5_GUN_STEP]
                                         : A.p.env[(long long)env * ENV_WORDS + W_STEP];
        const bool avail = ammo <= 0 || T.cooldown <= (double)cur_step - (double)own.w;
        double tx = mx, ty = my, tz = mz;
        if (avail) {
            double bd = 0; bool found = false;
            for (int i = T.n_lw; i < D; ++i) {
                if (!(A.p.flagw[b + i] & F_OFF)) continue;
                const V4<R> q = ld4(snap + b + i);
                const double dd = sq3((double)q.x - mx, (double)q.y - my, (double)q.z - mz);
                if (!found || dd < bd) { found = true; bd = dd; tx = q.x; ty = q.y; tz = q.z; }
            }
        } else {
            const V4<R> f = ld4(A.p.state + 12 * stride + s);
            tx = f.x; ty = f.y; tz = f.z;
        }
        const double vx = tx - mx, vy = ty - my, vz = tz - mz, n = norm3(vx, vy, vz);
        if (n > 0) { cmd[0] = vx / n; cmd[1] = vy / n; cmd[2] = vz / n; } else { cmd[0] = vx; cmd[1] = vy; cmd[2] = vz; }
        cmd[3] = T.bt_speed;
    };
    bool policy32 = false;                           // the command is the float32 array of an SB3 policy (see below)
    const int drv = (FAM == FAM_DRIVEN && is_lw) ? T.lw_driver[d] : DRV_LEGACY;
    if (FAM == FAM_DRIVEN && drv != DRV_LEGACY) {
        if (drv == DRV_BT) { bt_command(); driven = true; }
        else if (drv == DRV_STOP) { cmd[3] = 1.0; driven = true; }
        else {
            bool serve = true;
            if (drv == DRV_NN_ALLY) {                 // exp05: get_armed_pursuers()[1:]
                serve = false;
                for (int j = 0; j < d; ++j) serve |= (A.p.flagw[b + j] & F_ARMED) != 0;
            }
            if (serve) {
                const float4 a = reinterpret_cast<const float4*>(A.lw_actions)[(long long)env * T.n_lw + d];
                cmd[0] = a.x; cmd[1] = a.y; cmd[2] = a.z; cmd[3] = a.w; driven = true; policy32 = true;
            }
        }
    } else if (d == agent_slot && FAM != FAM_L5_MULTI && !(FAM == FAM_DRIVEN && T.eval_task)) {
        const float4 a = reinterpret_cast<const float4*>(A.actions)[env];
        cmd[0] = a.x; cmd[1] = a.y; cmd[2] = a.z; cmd[3] = a.w; driven = true;
    } else if (FAM == FAM_STAGE01) {
        // stage01: the idle wingman keeps its zero setpoint; the munition holds its spawn point in QuadX
        // mode 7 with setpoint (x, y, yaw 0, z) (level2/components/quadcopter_manager.py:166-179), see below
    } else if (FAM == FAM_STAGE02) {
        // stage02: munitions are driven with [0,0,0,0.5] (zero direction: hover) and drive_support_pursuers
        // loops over the invaders again, so the support wingman keeps its zero setpoint
        // (level3/components/quadcopter_manager.py:176-205)
    } else if (!is_lw) {
        // KamikazeNavigator.update: check_transition, then execute the state fetched BEFORE it
        const int nav = A.p.nav[s];
        int new_nav = nav;
        bool any_lw = false;
        for (int j = 0; j < T.n_lw; ++j) any_lw |= (A.p.flagw[b + j] & F_OFF) != 0;
        auto path_clear = [&](double degrees) {
            if (T.lm_nav == 0) return false;             // air_combat_only :87-96 always False
            const double abx = T.building[0] - mx, aby = T.building[1] - my, abz = T.building[2] - mz;
            const double nab = norm3(abx, aby, abz);
            for (int j = 0; j < T.n_lw; ++j) {
                if (!(A.p.flagw[b + j] & F_OFF)) continue;
                const V4<R> q = ld4(snap + b + j);
                const double apx = (double)q.x - mx, apy = (double)q.y - my, apz = (double)q.z - mz;
                const double nap = norm3(apx, apy, apz);
                if (nap > nab) continue;
                const double ang = acos((apx * abx + apy * aby + apz * abz) / (nap * nab)) * (180.0 / 3.141592653589793);
                if (ang <= degrees / 2) return false;     // a wingman sits inside the cone
            }
            return true;
        };
        double tx = 0, ty = 0, tz = 0; bool moving = false;
        if (nav == NAV_WAIT) {
            if (path_clear(60.0)) new_nav = NAV_BUILDING;
            else if (any_lw) new_nav = NAV_WINGMAN;
        } else if (nav == NAV_WINGMAN) {
            if (!any_lw) new_nav = NAV_BUILDING;
            double bd = 0; bool found = false;
            for (int j = 0; j < T.n_lw; ++j) {
                if (!(A.p.flagw[b + j] & F_OFF)) continue;
                const V4<R> q = ld4(snap + b + j);
                const double dd = sq3((double)q.x - mx, (double)q.y - my, (double)q.z - mz);
                if (!found || dd < bd) { found = true; bd = dd; tx = q.x; ty = q.y; tz = q.z; }
            }
            moving = true;
        } else {
            if (!path_clear(45.0)) new_nav = NAV_WINGMAN;
            tx = T.building[0]; ty = T.building[1]; tz = T.building[2]; moving = true;
        }
        if (new_nav != nav) A.p.nav[s] = (unsigned char)new_nav;
        if (moving) {
            const double vx = tx - mx, vy = ty - my, vz = tz - mz, n = norm3(vx, vy, vz);
            if (n > 0) { cmd[0] = vx / n; cmd[1] = vy / n; cmd[2] = vz / n; } else { cmd[0] = vx; cmd[1] = vy; cmd[2] = vz; }
        }
        cmd[3] = T.lm_speed; driven = true;
    } else {
        // drive_loyalwingmen: get_armed_pursuers()[1:]; level5: get_allies(armed=True) = every wingman but the agent
        int armed_before = fam_l5(FAM) ? 1 : 0;
        for (int j = 0; j < d; ++j) armed_before += (A.p.flagw[b + j] & F_ARMED) ? 1 : 0;
        if (armed_before >= 1) {
            if (T.ally_mode == 1) { cmd[3] = T.ally_stop; }
            else bt_command();
            driven = true;
        }
    }
    if (FAM == FAM_L5_MULTI && is_lw && driven && A.mo_last_action)     // Quadcopter.last_action (quadcopter.py:415-419) = the teacher action
        reinterpret_cast<float4*>(A.mo_last_action)[(long long)env * T.n_lw + d] =
            make_float4((float)cmd[0], (float)cmd[1], (float)cmd[2], (float)cmd[3]);
    R sp[4] = {0, 0, 0, 0};
    if (FAM == FAM_DRIVEN && policy32) {
        // convert_command_to_setpoint on the float32 array predict() returns: numpy keeps norm, division and product in
        // float32 (quadcopter.py:391-396); the setpoint array itself is float64
        const float cx = (float)cmd[0], cy = (float)cmd[1], cz = (float)cmd[2], cm = (float)cmd[3];
        const float n = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(cx, cx), __fmul_rn(cy, cy)), __fmul_rn(cz, cz)));
        const float dn = n > 0.f ? n : 1.f;
        sp[0] = (R)__fmul_rn(cm, __fdiv_rn(cx, dn)); sp[1] = (R)__fmul_rn(cm, __fdiv_rn(cy, dn));
        sp[2] = 0; sp[3] = (R)__fmul_rn(cm, __fdiv_rn(cz, dn));
    } else
    if (driven) {                                   // convert_command_to_setpoint quadcopter.py:379-396
        const double n = norm3(cmd[0], cmd[1], cmd[2]);
        const double dn = n > 0 ? n : 1.0;
        sp[0] = (R)(cmd[3] * (cmd[0] / dn)); sp[1] = (R)(cmd[3] * (cmd[1] / dn));
        sp[2] = 0; sp[3] = (R)(cmd[3] * (cmd[2] / dn));
    }

    const bool mode7 = FAM == FAM_STAGE01 && !is_lw;
    if (mode7) {
        const V4<R> f = ld4(A.p.state + 12 * stride + s);           // replace() stored the hold point here
        sp[0] = f.x; sp[1] = f.y; sp[2] = 0; sp[3] = f.z;
    }
    // ---- dynamic state: 16-byte loads (quads 0..9), 16 substeps in registers, write-back ------------
    Drone<R> st;
    V4<R>* gp = A.p.state + s;
    Words::load(st, gp, stride);
    Imu<R> imu;
    const uint32_t env_id = T.env_offset + (uint32_t)env;
    const uint32_t phys0 = (uint32_t)A.p.env[(long long)env * ENV_WORDS + W_PHYS_CTR];
    if (FAM == FAM_STAGE01) {
        // replace_invader ends with one update_imu/update_control/update_physics outside the stepping loop:
        // PID and motors advance once more and the applied force is still pending at the next
        // stepSimulation, i.e. it adds to the first substep (quadcopter_manager.py:176-179)
        Wrench<R> extra{0, 0, 0, 0, 0, 0};
        const int fw = A.p.flagw[s];
        const int owed = ((fw & F_PENDING) ? 1 : 0) + ((fw & F_PENDING2) ? 1 : 0);
        for (int n = 0; n < owed; ++n) {
            const Wrench<R> W = quad_forces<R, NOISE>(st, sp, mode7, A.q, imu, T.k0, T.k1, env_id, (uint32_t)d, phys0,
                                                      quat_rot(st.qx, st.qy, st.qz, st.qw));
            extra.fx += W.fx; extra.fy += W.fy; extra.fz += W.fz; extra.tx += W.tx; extra.ty += W.ty; extra.tz += W.tz;
        }
        for (int k = 0; k < T.substeps; ++k) {
            const Rot<R> M = quat_rot(st.qx, st.qy, st.qz, st.qw);
            Wrench<R> W = quad_forces<R, NOISE>(st, sp, mode7, A.q, imu, T.k0, T.k1, env_id, (uint32_t)d, phys0 + (uint32_t)k, M);
            if (k == 0) { W.fx += extra.fx; W.fy += extra.fy; W.fz += extra.fz; W.tx += extra.tx; W.ty += extra.ty; W.tz += extra.tz; }
            quad_integrate<R>(st, W, A.q, M);
        }
    } else if constexpr (sizeof(R) == 4) {
        // only the IMU record of the last substep is read: the others run without materialising it
        const int last = T.substeps - 1;
        for (int k = 0; k < last; ++k)
            quad_substep_f32<NOISE, BUILTIN, false>(st, sp, A.q, imu, A.rk, env_id, (uint32_t)d, phys0 + (uint32_t)k);
        quad_substep_f32<NOISE, BUILTIN, true>(st, sp, A.q, imu, A.rk, env_id, (uint32_t)d, phys0 + (uint32_t)last);
    } else {
        for (int k = 0; k < T.substeps; ++k)
            quad_substep<R, NOISE>(st, sp, A.q, imu, T.k0, T.k1, env_id, (uint32_t)d, phys0 + (uint32_t)k);
    }
    asm volatile("griddepcontrol.launch_dependents;");      // env_kernel's blocks may be placed while the state drains
    st4(A.p.imu[par ^ 1] + s, V4<R>{imu.px, imu.py, imu.pz, own.w});
    constexpr bool REC_PER_LW = fam_l5(FAM) || FAM == FAM_DRIVEN;     // an imu record per wingman (TaskParams::n_rec)
    if (REC_PER_LW ? is_lw : d == 0) {
        V4<R>* ag = reinterpret_cast<V4<R>*>(A.p.agent + ((long long)env * T.n_rec + (REC_PER_LW ? d : 0)) * AG_WORDS);
        st4(ag, V4<R>{imu.ub, imu.vb, imu.wb, imu.roll});
        st4(ag + 1, V4<R>{imu.pitch, quat_yaw(imu.qx, imu.qy, imu.qz, imu.qw), imu.p, imu.q});
        st4(ag + 2, V4<R>{imu.r, imu.qx, imu.qy, imu.qz});
        st4(ag + 3, V4<R>{imu.qw, 0, 0, 0});
    }
    Words::store(st, gp, stride);
    DC_TL_END(A.tl_slot);
}

// ================================================================================================
// env_kernel
// ================================================================================================
// Shared-memory view of one block (NS = EPB * D slots).
template <typename R> struct Smem {
    R* imu;         // [NS][3] imu position of this step (state before the last substep)
    R* newpos;      // [NS][3] teleport target written by the env pass (or the spawn job: Philox base, n, i)
    R* last;        // [NS] last_fired_step
    int* ev;        // [NS] EV_*
    int* ammo;      // [NS]
    int* list;      // [NS] per warp: armed slots for the next step, then the entities to project
    int* envflag;   // [EPB]
    double* rn;     // [NS] LiDAR: normalised distance of the projection (float64, the winner test needs it)
    int* cell;      // [NS] LiDAR: cell index of the projection, -1 = none
    double* ang;    // [NS][2] level5 only: (theta, phi) of the projection, kept as features
};

template <typename R>
__device__ __forceinline__ Smem<R> carve_smem(unsigned char* base, int ns, int epb, bool level5) {
    Smem<R> s;
    size_t off = 0;
    auto take = [&](size_t bytes) { void* p = base + off; off += (bytes + 15) & ~size_t(15); return p; };
    s.rn = (double*)take(sizeof(double) * ns);
    s.newpos = (R*)take(sizeof(R) * 3 * ns);
    s.imu = (R*)take(sizeof(R) * 3 * ns);
    s.last = (R*)take(sizeof(R) * ns);
    s.ev = (int*)take(sizeof(int) * ns);
    s.ammo = (int*)take(sizeof(int) * ns);
    s.list = (int*)take(sizeof(int) * ns);
    s.envflag = (int*)take(sizeof(int) * epb);
    s.cell = (int*)take(sizeof(int) * ns);
    s.ang = level5 ? (double*)take(sizeof(double) * 2 * ns) : nullptr;
    return s;
}

inline size_t smem_bytes(int ns, int epb, size_t sizeofR, bool level5) {
    auto up = [](size_t b) { return (b + 15) & ~size_t(15); };
    return up(8 * (size_t)ns) + 2 * up(sizeofR * 3 * ns) + up(sizeofR * ns) + 4 * up(4 * ns) + up(4 * epb) + (level5 ? up(16 * (size_t)ns) : 0);
}

// ------------------------------------------------------------------------------------------------
// Env-pass helpers.  `b` = index of the env's slot 0 inside the block's shared arrays.
// ------------------------------------------------------------------------------------------------
// generate_positions(n, r)[i]  exp02_vFinal_task.py:583-607 (thetas drawn first, then phis); Philox SPAWN stream.
__device__ __forceinline__ void spawn_point_core(uint32_t k0, uint32_t k1, uint32_t env_id, uint32_t i_theta, uint32_t i_phi,
                                              double r, double lo, double* out) {
    const double PI = 3.141592653589793;
    const double theta = 0.0 + (PI - 0.0) * philox_uniform(k0, k1, env_id, STREAM_SPAWN, i_theta);
    const double phi = lo + (PI / 2 - lo) * philox_uniform(k0, k1, env_id, STREAM_SPAWN, i_phi);
    double sp, cp, st, ct;
    sincos(phi, &sp, &cp); sincos(theta, &st, &ct);
    out[0] = r * sp * ct;
    out[1] = r * sp * st;
    out[2] = r * cp;
}
__device__ __forceinline__ void spawn_point(const TaskParams& T, uint32_t env_id, uint32_t base, int n, int i, double r, double* out) {
    const double min_z = 4.0;
    double lo;
    if (r == T.born) lo = T.acos_born;
    else if (r == T.lw_spawn) lo = T.acos_lw;
    else lo = (r >= min_z) ? acos(fmin(min_z, r) / r) : 0.0;
    spawn_point_core(T.k0, T.k1, env_id, base + i, base + n + i, r, lo, out);
}
// one uniform of the HIT stream (Gun.shoot's random.random(), gun.py:86-99)
__device__ __forceinline__ double hit_uniform(uint32_t k0, uint32_t k1, uint32_t env_id, uint32_t idx) {
    return philox_uniform(k0, k1, env_id, STREAM_HIT, idx);
}

// GS > 1 (stage03 family, envs with many drones): the env pass gives every env a GROUP of GS lanes instead of one lane.
// All lanes of a group run the same sequential logic on the same data (the scalars live replicated in their registers,
// stores of identical values to shared memory are idempotent), and the O(drones) loops -- nearest-in-range, outside-dome
// counts, wave set-up, offsets refresh, spawn draws -- are strided over the group with shuffle reductions.  A swarm env
// (68 drones, 4 envs per warp) ran them in 4 of 32 lanes otherwise.
template <typename R, int FAM, int GS = 1> struct EnvCtx {
    const TaskParams& T;
    Smem<R>& S;
    int b, le;
    uint32_t env_id;         // global env index (Philox counter word)
    int32_t* w;              // env scalar words (local copy)
    double inv_dome;         // 1 / dome radius: the position scale of normalize_inertial_data
    // level5: Gun.current_step == Task.current_step (gun.py:44-47, level5_c1_fusion_task.py:74-76).  The env
    // broadcasts the step as publisher 0 (level5_envrionment.py:276-281) and the first munition is body 0 (spawned
    // before the ground plane), so every disarm of that munition makes MessageHub.terminate(0) re-broadcast
    // {"termination": True} on the step topic (message_hub.py:56-65): all guns and the task read step 0 until the
    // next broadcast.
    int agent = 0, gun_step = 0;
    bool registered = false;
    int32_t* w5 = nullptr;           // level5: this env's row of SimPtrs::env5
    int32_t* kills = nullptr;        // FAM_DRIVEN: this env's row of SimPtrs::lw_kills
    int g = 0;                       // lane within the env's group, and the group's lane mask (GS > 1)
    unsigned gmask = 0xffffffffu;
    __device__ void gsync() const { if (GS > 1) __syncwarp(gmask); }
    __device__ int gsum(int v) const {
        if (GS > 1) for (int o = GS / 2; o > 0; o >>= 1) v += __shfl_xor_sync(gmask, v, o);
        return v;
    }
    __device__ bool gany(bool p) const { return GS > 1 ? (__ballot_sync(gmask, p) & gmask) != 0 : p; }
    // lexicographic (distance, index) minimum over the group: the ascending scan with a strict '<' keeps the first index
    __device__ void gargmin(int& best, double& bd) const {
        if (GS > 1) for (int o = GS / 2; o > 0; o >>= 1) {
            const int ob = __shfl_xor_sync(gmask, best, o);
            const double od = __shfl_xor_sync(gmask, bd, o);
            if (ob >= 0 && (best < 0 || od < bd || (od == bd && ob < best))) { best = ob; bd = od; }
        }
    }
    __device__ EnvCtx(const TaskParams& t, Smem<R>& s, int base, int local_env, uint32_t id, int32_t* words)
        : T(t), S(s), b(base), le(local_env), env_id(id), w(words), inv_dome(1.0 / t.dome) {}
    __device__ int gstep() const { return fam_l5(FAM) ? gun_step : w[W_STEP]; }
    __device__ void broadcast_step() { gun_step = w[W_STEP]; registered = true; }

    __device__ void disarm(int d) {                       // Quadcopter.disarm quadcopter.py:461-478
        S.ev[b + d] = (S.ev[b + d] & ~(EV_LIVE | EV_SNAP)) | EV_ZEROED;
        if (fam_l5(FAM) && d == T.n_lw && registered) { gun_step = 0; registered = false; }
    }
    __device__ void arm(int d) {                          // Quadcopter.arm quadcopter.py:445-459 (gun.reset())
        S.ev[b + d] = (S.ev[b + d] & ~EV_SNAP) | EV_LIVE | EV_REARMED;
        S.ammo[b + d] = d >= T.n_lw ? 10 : (FAM == FAM_STAGE02 && d > 0) ? T.support_munition : T.munition;
        S.last[b + d] = (R)(-T.cooldown);
    }
    __device__ void replace(int d, double x, double y, double z) {   // quadcopter.py:433-439
        S.ev[b + d] = (S.ev[b + d] & ~EV_SPAWNJOB) | EV_REPLACED;
        S.newpos[3 * (b + d) + 0] = (R)x; S.newpos[3 * (b + d) + 1] = (R)y; S.newpos[3 * (b + d) + 2] = (R)z;
    }
    __device__ bool live(int d) const { return S.ev[b + d] & EV_LIVE; }
    __device__ bool off(int d) const { return S.ev[b + d] & EV_OFF; }
    __device__ double spawn_u(uint32_t idx) const { return philox_uniform(T.k0, T.k1, env_id, STREAM_SPAWN, idx); }
    __device__ void gen_position(uint32_t base, int n, int i, double r, double* out) const { spawn_point(T, env_id, base, n, i, r, out); }
    // A munition wave is spawned by the warp, one lane per munition, after the env pass (env_kernel "spawn pass"): the
    // env pass only leaves the job (Philox counter base, n, i) in the slot's newpos words.  A wave of k positions would
    // otherwise be k x ~500 dependent instructions in ONE lane while the other 31 lanes of the warp -- and, at the
    // end of the kernel, the whole GPU -- wait for it.
    __device__ void spawn_job(int d, uint32_t base, int n, int i) {
        S.ev[b + d] |= EV_REPLACED | EV_SPAWNJOB;
        int* jp = reinterpret_cast<int*>(S.newpos + 3 * (b + d));
        jp[0] = (int)base; jp[1] = n; jp[2] = i;
    }
    // stage02 generate_positions(n, r, r_max)[i]  level3/components/stages.py:350-368 (radius, theta, phi draws)
    __device__ void gen3(uint32_t base, int n, int i, double r, double r_max, double* out) const {
        const double PI = 3.141592653589793;
        if (r > r_max) r_max = r;
        const double radius = r + (r_max - r) * spawn_u(base + i);
        const double theta = 0.0 + (2 * PI - 0.0) * spawn_u(base + n + i);
        const double phi = 0.0 + (PI / 2 - 0.0) * spawn_u(base + 2 * n + i);
        out[0] = radius * sin(phi) * cos(theta);
        out[1] = radius * sin(phi) * sin(theta);
        out[2] = radius * cos(phi);
    }
    // stage01: np.random.uniform(-1, 1, 3) (pyflyt_level2_environment_modified_v2.py:48,85-100,153)
    __device__ void u3(double* out) {
        const uint32_t base = (uint32_t)w[W_SPAWN_CTR];
        for (int k = 0; k < 3; ++k) out[k] = -1.0 + (1.0 - -1.0) * spawn_u(base + k);
        w[W_SPAWN_CTR] += 3;
    }
    __device__ void replace_invader_stage01(int lm, const double* p) {   // level2 quadcopter_manager.py:166-179
        replace(lm, p[0], p[1], p[2]);
        S.ev[b + lm] |= (S.ev[b + lm] & EV_PENDING) ? EV_PENDING2 : EV_PENDING;   // caught on the terminal step: two owed
    }
    __device__ void reset_words() {                       // the episode counters of Env.reset
        w[W_STEP] = 0; w[W_MAX_STEP] = T.max_step;
        w[W_AGENT_KILLS] = w[W_ALLIES_KILLS] = w[W_DEADS] = 0; w[W_BUILDING] = 1;
        w[W_EP_RETURN] = __float_as_int(0.0f); w[W_EP_STEPS] = 0;
    }
    __device__ void reset_env_stage01() {                 // pyflyt_level2_environment_modified_v2.py:70-104
        reset_words();
        const int lm = T.n_lw;
        double p[3];
        u3(p); replace_invader_stage01(lm, p);
        u3(p); replace(0, p[0], p[1], p[2]);
        u3(p); replace(1, p[0], p[1], p[2]);
        set_last_closest(norm3((double)S.newpos[3 * (b + lm)] - (double)S.newpos[3 * b], (double)S.newpos[3 * (b + lm) + 1] - (double)S.newpos[3 * b + 1],
                               (double)S.newpos[3 * (b + lm) + 2] - (double)S.newpos[3 * b + 2]));
    }
    __device__ void env_init_stage01() {                  // :27-68: munition at p, agent at -p, idle wingman at (3,3,3)
        double p[3];
        u3(p);
        replace(T.n_lw, p[0], p[1], p[2]); replace(0, -p[0], -p[1], -p[2]); replace(1, 3.0, 3.0, 3.0);
        for (int d = 0; d < T.D; ++d) arm(d);
        refresh_offsets();
        w[W_INIT] = 1;
    }
    __device__ int row0() const {                         // distances[0]: first armed pursuer of the snapshot
        for (int j = 0; j < T.n_lw; ++j) if (off(j)) return j;
        return -1;
    }
    // stage02 Stage.on_episode_start (stages.py:110-124): arm everything, snapshot, last offsets := current
    __device__ void episode_start_stage02(double* last_dist) {
        for (int d = 0; d < T.D; ++d) arm(d);
        refresh_offsets();
        // distances agent -> munitions at the positions just assigned by replace()
        for (int i = 0; i < T.n_lm; ++i) {
            const int a = b, c = b + T.n_lw + i;
            last_dist[i] = norm3((double)S.newpos[3 * a] - (double)S.newpos[3 * c], (double)S.newpos[3 * a + 1] - (double)S.newpos[3 * c + 1],
                                 (double)S.newpos[3 * a + 2] - (double)S.newpos[3 * c + 2]);
        }
    }
    // stage02 placement: munitions on r in U(r0, r1), wingmen on r in U(1, 1), then Stage.on_episode_start
    __device__ void place_stage02(double r0, double r1, double* last_dist) {
        uint32_t base = (uint32_t)w[W_SPAWN_CTR];
        for (int i = 0; i < T.n_lm; ++i) { double p[3]; gen3(base, T.n_lm, i, r0, r1, p); replace(T.n_lw + i, p[0], p[1], p[2]); }
        w[W_SPAWN_CTR] += 3 * T.n_lm;
        base = (uint32_t)w[W_SPAWN_CTR];
        for (int j = 0; j < T.n_lw; ++j) { double p[3]; gen3(base, T.n_lw, j, 1.0, 0.0, p); replace(j, p[0], p[1], p[2]); }
        w[W_SPAWN_CTR] += 3 * T.n_lw;
        episode_start_stage02(last_dist);
    }
    __device__ void env_init_stage02(double* last_dist) {  // stages.py:96-100,378-397
        place_stage02(2.0, 0.0, last_dist);
        w[W_INIT] = 1;
    }
    __device__ void reset_env_stage02(double* last_dist) { // stages.py:102-135
        reset_words();
        for (int d = 0; d < T.D; ++d) disarm(d);
        place_stage02(T.respawn_r0, T.respawn_r1, last_dist);
    }
    __device__ void setup_round(int k) {                  // exp02_vFinal_task.py:179-195
        for (int i = g; i < T.n_lm; i += GS) disarm(T.n_lw + i);
        gsync();
        const uint32_t base = (uint32_t)w[W_SPAWN_CTR];
        for (int i = g; i < k; i += GS) {
            spawn_job(T.n_lw + i, base, k, i);
            arm(T.n_lw + i);
        }
        gsync();
        w[W_SPAWN_CTR] += 2 * k;
    }
    // advance_round (stage03 :154-174, level5 :139-152): the next wave once the munitions of this one are gone
    __device__ void advance_round() {
        const int last = fam_l5(FAM) ? T.max_rounds : T.n_lm;
        w[W_ROUND] += (w[W_ROUND] < last) ? 1 : last;
        if (fam_l5(FAM)) setup_round5(w[W_ROUND]); else setup_round(w[W_ROUND]);
        refresh_offsets();
        S.envflag[le] |= EF_NAV_RESET;
    }
    __device__ void refresh_offsets() {                   // OffsetHandler.on_episode_start: snapshot := live set
        gsync();
        for (int d = g; d < T.D; d += GS) {
            int e = S.ev[b + d];
            S.ev[b + d] = (e & EV_LIVE) ? (e | EV_OFF) : (e & ~EV_OFF);
        }
        gsync();
    }
    __device__ void episode_start(double* lw_init) {      // exp02_vFinal_task.py:258-267, level5 :262-273
        w[W_ROUND] = T.initial_round;
        if (fam_l5(FAM)) setup_round5(T.initial_round); else setup_round(T.initial_round);
        for (int j = g; j < T.n_lw; j += GS) arm(j);
        gsync();
        const bool fixed = !fam_l5(FAM) && T.fixed_lw_spawn;
        const uint32_t base = (uint32_t)w[W_SPAWN_CTR];
        for (int j = g; j < T.n_lw; j += GS) {
            double p[3];
            if (fixed) { p[0] = lw_init[3 * j]; p[1] = lw_init[3 * j + 1]; p[2] = lw_init[3 * j + 2]; }
            else gen_position(base, T.n_lw, j, T.lw_spawn, p);
            replace(j, p[0], p[1], p[2]);
        }
        gsync();
        if (!fixed) w[W_SPAWN_CTR] += 2 * T.n_lw;
    }
    // Env.__init__: Task.on_env_init + on_episode_start  exp02_vFinal_environment.py:62-63, task :248-252,622-646
    // (level5: on_env_init :253-257,609-660 + set_agent())
    __device__ void env_init(double* lw_init) {
        uint32_t base = (uint32_t)w[W_SPAWN_CTR];
        for (int i = g; i < T.n_lm; i += GS) {
            double p[3];
            gen_position(base, T.n_lm, i, T.born, p);
            replace(T.n_lw + i, p[0], p[1], p[2]);
        }
        w[W_SPAWN_CTR] += 2 * T.n_lm;
        base = (uint32_t)w[W_SPAWN_CTR];
        for (int j = g; j < T.n_lw; j += GS) {
            double p[3];
            gen_position(base, T.n_lw, j, T.lw_spawn, p);
            if (!fam_l5(FAM)) { lw_init[3 * j] = p[0]; lw_init[3 * j + 1] = p[1]; lw_init[3 * j + 2] = p[2]; }
            replace(j, p[0], p[1], p[2]);
        }
        if (GS > 1) __threadfence_block();                 // episode_start of the other lanes reads lw_init (fixed spawn)
        gsync();
        w[W_SPAWN_CTR] += 2 * T.n_lw;
        if (fam_l5(FAM)) {
            if (FAM == FAM_L5_MULTI && T.l5_eval) agent = 0;                        // Teacher_Student=False: no agent is chosen, no draw
            else {
                agent = (int)(spawn_u((uint32_t)w[W_SPAWN_CTR]) * T.n_lw); // entities_manager.py:350-383, randomness as data
                w[W_SPAWN_CTR] += 1;
            }
            registered = false;
        }
        episode_start(lw_init);
        w[W_INIT] = 1;
    }
    // Env.reset -> Task.on_reset  exp02_vFinal_environment.py:133-151, task :254-273 (level5_envrionment.py:203-231,
    // task on_reset :275-283)
    __device__ void reset_env(double* lw_init) {
        if (FAM == FAM_DRIVEN && kills) for (int j = 0; j < T.n_lw; ++j) kills[j] = 0;      // on_episode_start evaluation_task.py:360-364
        reset_words();
        set_last_closest(T.dome);
        for (int d = g; d < T.D; d += GS) disarm(d);
        gsync();
        episode_start(lw_init);
        refresh_offsets();
        S.envflag[le] |= EF_NAV_RESET;
        if (fam_l5(FAM)) broadcast_step();                 // reset_step_counter: step 0
    }
    // ---- level5 (Level5C1FusionTask) ----
    // ---- level5 (Level5C1FusionTask) ----
    __device__ int n_active(int k) const {                // setup_round :158-160
        const int n = (k - 1) * T.invaders_per_round + T.initial_invaders;
        return n < T.n_lm ? n : T.n_lm;
    }
    __device__ void setup_round5(int k) {                 // level5_c1_fusion_task.py:154-169
        for (int i = 0; i < T.n_lm; ++i) disarm(T.n_lw + i);
        const int n = n_active(k);
        const uint32_t base = (uint32_t)w[W_SPAWN_CTR];
        for (int i = 0; i < n; ++i) {
            spawn_job(T.n_lw + i, base, n, i);
            arm(T.n_lw + i);
        }
        w[W_SPAWN_CTR] += 2 * n;
    }
    // ---- the family's Env.__init__ and Env.reset ----
    __device__ void init_task(double* lw_init, double* last_dist) {
        for (int k = 0; k < ENV_WORDS; ++k) w[k] = 0;
        if (fam_l5(FAM)) {
            for (int k = 0; k < ENV5_WORDS; ++k) w5[k] = 0;
            w5[W5_LAST_DIST_LO] = 0; w5[W5_LAST_DIST_HI] = 0x7ff80000;     // NaN: last_distance not set yet
        }
        if (FAM == FAM_STAGE01) env_init_stage01(); else if (FAM == FAM_STAGE02) env_init_stage02(last_dist); else env_init(lw_init);
    }
    __device__ void reset_task(double* lw_init, double* last_dist) {
        if (FAM == FAM_STAGE01) reset_env_stage01(); else if (FAM == FAM_STAGE02) reset_env_stage02(last_dist); else reset_env(lw_init);
        if (fam_l5(FAM)) { w5[W5_STACK_MODE] = STACK_EMPTY; w5[W5_OBS_CALL] += T.l5_base ? 3 : 1; }
    }
    __device__ void set_last_closest(double v) {
        long long bits = __double_as_longlong(v);
        w[W_LAST_CLOSEST_LO] = (int32_t)(bits & 0xffffffffLL); w[W_LAST_CLOSEST_HI] = (int32_t)(bits >> 32);
    }
    __device__ double last_closest() const {
        long long bits = ((long long)w[W_LAST_CLOSEST_HI] << 32) | (unsigned int)w[W_LAST_CLOSEST_LO];
        return __longlong_as_double(bits);
    }
    __device__ double pos(int d, int k) const { return (double)S.imu[3 * (b + d) + k]; }
    __device__ double dist2(int a, int c) const {
        return sq3(pos(a, 0) - pos(c, 0), pos(a, 1) - pos(c, 1), pos(a, 2) - pos(c, 2));
    }
    // Gun.is_available gun.py:56-75 (current_step == env step after the broadcast)
    __device__ bool gun_available(int j) const {
        if (S.ammo[b + j] <= 0) return true;
        return T.cooldown <= (double)gstep() - (double)S.last[b + j];
    }
    __device__ void gun_state(int j, float* g) const {      // Gun.get_state gun.py:101-113
        const double wait = fmax(T.cooldown - ((double)gstep() - (double)S.last[b + j]), 0.0);
        const int mx = T.munition > 0 ? T.munition : 1;
        g[0] = (float)((double)S.ammo[b + j] / (double)mx);
        g[1] = (float)(wait / T.cooldown);
        g[2] = gun_available(j) ? 1.f : 0.f;
    }
    // identify_invaders_in_range(...)[j][0] (offsets_handler.py:283-309: ascending stable sort -> first index wins ties; sqrt is
    // monotone, so squared distances pick the same winner).
    // Both engagement passes of a step read the SAME stale distance matrix (positions and snapshot membership do not change
    // between them), so for every pursuer the shoot-range and the explosion-range candidate is the same nearest snapshot
    // invader, in range or not: found once per step and parked in S.cell (free until P4) with the two range bits.
    __device__ void nearest_all() {
        const double s2 = T.shoot * T.shoot, e2 = T.expl * T.expl;
        for (int j = 0; j < T.n_lw; ++j) {
            int code = -1;
            if (off(j)) {
                int best = -1; double bd = 0.0;
                for (int i = T.n_lw + g; i < T.D; i += GS) {
                    if (!off(i)) continue;
                    const double d = dist2(j, i);
                    if (best < 0 || d < bd) { best = i; bd = d; }
                }
                gargmin(best, bd);
                if (best >= 0) code = best | (bd < s2 ? 1 << 16 : 0) | (bd < e2 ? 1 << 17 : 0);
            }
            S.cell[b + j] = code;
        }
    }
    __device__ int nearest_shoot(int j) const { const int c = S.cell[b + j]; return (c >= 0 && (c & (1 << 16))) ? (c & 0xffff) : -1; }
    __device__ int nearest_expl(int j) const { const int c = S.cell[b + j]; return (c >= 0 && (c & (1 << 17))) ? (c & 0xffff) : -1; }
    // identify_closest_invader(src) offsets_handler.py:256-281 (np.argmin: first index on ties)
    __device__ int nearest_invader(int src) const {
        int best = -1; double bd = 0.0;
        for (int i = T.n_lw + g; i < T.D; i += GS) {
            if (!off(i)) continue;
            const double d = dist2(src, i);
            if (best < 0 || d < bd) { best = i; bd = d; }
        }
        gargmin(best, bd);
        return best;
    }
    // identify_closest_ally(as) on the offsets snapshot (the agent itself when it flies alone), then that ally's nearest
    // invader; -1 when the agent is not in the snapshot
    __device__ int ally_target(int as) const {
        int src = -1;
        if (off(as)) {
            int n_all = 0;
            for (int j = 0; j < T.n_lw; ++j) n_all += off(j) ? 1 : 0;
            if (n_all <= 1) src = as;
            else {
                double bd = 0;
                for (int j = 0; j < T.n_lw; ++j) {
                    if (j == as || !off(j)) continue;
                    const double dd = dist2(j, as);
                    if (src < 0 || dd < bd) { src = j; bd = dd; }
                }
            }
        }
        return src >= 0 ? nearest_invader(src) : -1;
    }
    __device__ int count_outside_dome(int lo, int hi) const {
        int n = 0;
        const double r2 = T.dome * T.dome;
        for (int d = lo + g; d < hi; d += GS)
            if (off(d) && sq3(pos(d, 0), pos(d, 1), pos(d, 2)) > r2) ++n;
        return gsum(n);
    }
};

// Appends the values of the lanes whose predicate holds to list[n_before..) in lane order and returns the
// new length.  Must be called by all 32 lanes of the warp; the list is private to the warp.
__device__ __forceinline__ int warp_compact(bool pred, int value, int* list, int n_before) {
    const unsigned m = __ballot_sync(0xffffffffu, pred);
    if (pred) list[n_before + __popc(m & ((1u << (threadIdx.x & 31)) - 1))] = value;
    return n_before + __popc(m);
}

#ifdef DC_PROFILE_PHASES      // per-warp clock stamps at the phase borders of env_kernel (profiles/phase_clocks.py)
__device__ long long g_phase_clk[8192 * 8];
#define DC_STAMP_STEP(k) do { if ((threadIdx.x & 31) == 0) { const int gw = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); if (gw < 8192) g_phase_clk[gw * 8 + (k)] = clock64(); } } while (0)
#else
#define DC_STAMP_STEP(k) do { } while (0)
#endif
#define DC_STAMP(k) do { if (MODE == MODE_STEP) DC_STAMP_STEP(k); } while (0)      // reset launches stamp nothing

// ------------------------------------------------------------------------------------------------
// P3 per family: what each reference task does in Task.on_step_middle (engagement, reward, termination) and
// Task.on_step_end.  env_kernel's env loop calls the family's pair and writes the outputs common to all families.
// ------------------------------------------------------------------------------------------------
// normalize_inertial_data's clip(v / scale, -1, 1).  The float32 build multiplies in float32 (its inputs are float32
// state; one rounding of difference at most), the float64 build keeps the reference's float64 arithmetic.
template <typename R> __device__ __forceinline__ float nrm(double v, double inv_scale) {
    if constexpr (sizeof(R) == 4) return fminf(fmaxf((float)v * (float)inv_scale, -1.0f), 1.0f);
    else return (float)fmin(fmax(v * inv_scale, -1.0), 1.0);
}
// the scales of normalize_inertial_data normalization.py:6-110 (the position scale is the dome radius)
constexpr double INV_SPEED = 1.0 / (1 * 10 * (1000.0 / 3600.0));
constexpr double INV_PI = 1.0 / 3.141592653589793, INV_2PI = 1.0 / (2 * 3.141592653589793);

// What on_step_middle hands to the rest of the step.
struct StepMiddle {
    double reward = 0.0;
    bool done = false, lm_alive = false, lw_alive = false, all_over = false;
    bool caught = false;     // stage01: the munition was caught
    float g[3];              // the agent's Gun.get_state
};

// ================= stage01: compute_reward / compute_termination (level2 modified_v2 :157-191) =================
template <typename R, int FAM, int GS> __device__ __forceinline__ StepMiddle stage01_on_step_middle(EnvCtx<R, FAM, GS>& C, const R* ag, const double* ap) {
    const TaskParams& T = C.T;
    int32_t* w = C.w;
    StepMiddle m;
    const int lm = T.n_lw;
    const double dcur = sqrt(C.dist2(lm, 0));
    double bonus = 0, penalty = 0;
    if (dcur < C.last_closest()) bonus += 10.0 * norm3((double)ag[AG_UB], (double)ag[AG_VB], (double)ag[AG_WB]);
    m.caught = dcur < 0.4;                           // CATCH_DISTANCE (:34)
    if (m.caught) bonus += 1000.0;
    if (dcur > T.dome) penalty += 1000.0;
    m.reward = -dcur + bonus - penalty;
    m.done = w[W_STEP] > w[W_MAX_STEP];
    m.done |= norm3(ap[0], ap[1], ap[2]) > T.dome;
    m.done |= norm3(C.pos(lm, 0), C.pos(lm, 1), C.pos(lm, 2)) > T.dome;
    C.gun_state(C.agent, m.g);
    C.set_last_closest(dcur);
    return m;
}
// replace_invader_if_close + update_last_distance (:148-155,193-198)
template <typename R, int FAM, int GS> __device__ __forceinline__ void stage01_on_step_end(EnvCtx<R, FAM, GS>& C, const StepMiddle& m, const double* ap) {
    if (m.caught) {
        const int lm = C.T.n_lw, b = C.b;
        double p[3];
        C.w[W_AGENT_KILLS] += 1;
        C.u3(p);
        C.replace_invader_stage01(lm, p);
        C.set_last_closest(norm3((double)C.S.newpos[3 * (b + lm)] - ap[0], (double)C.S.newpos[3 * (b + lm) + 1] - ap[1],
                                 (double)C.S.newpos[3 * (b + lm) + 2] - ap[2]));
    }
}

// ================= stage02: L3Stage1.on_step_middle (level3/components/stages.py:144-179) =================
template <typename R, int FAM, int GS> __device__ __forceinline__ StepMiddle stage02_on_step_middle(EnvCtx<R, FAM, GS>& C, const R* ag, const double* last_dist) {
    const TaskParams& T = C.T;
    Smem<R>& S = C.S;
    int32_t* w = C.w;
    const int b = C.b, D = T.D;
    StepMiddle m;
    int shots = 0, exploded = 0;
    C.nearest_all();
    for (int j = 0; j < T.n_lw; ++j) {              // process_shoot_range_invaders + shoot_by_ids (quadcopter_manager.py:155-169)
        if (!C.off(j)) continue;
        const int tgt = C.nearest_shoot(j);
        if (tgt < 0) continue;
        if (S.ammo[b + j] == 0) { C.disarm(tgt); ++shots; continue; }      // "LW suicided to kill LM"
        if (!C.gun_available(j)) continue;
        S.ammo[b + j] -= 1; S.last[b + j] = (R)w[W_STEP];
        const double u = hit_uniform(T.k0, T.k1, C.env_id, (uint32_t)w[W_HIT_CTR]);
        w[W_HIT_CTR] += 1;
        if (u < T.fire_p) { C.disarm(tgt); ++shots; }
    }
    for (int j = 0; j < T.n_lw; ++j) {              // process_explosion_range_invaders
        if (!C.off(j)) continue;
        const int tgt = C.nearest_expl(j);
        if (tgt < 0) continue;
        C.disarm(j); C.disarm(tgt); ++exploded;
    }
    w[W_AGENT_KILLS] += shots; w[W_DEADS] += exploded;
    C.gun_state(C.agent, m.g);
    // compute_reward stages.py:234-296 with the closest distances of OffsetHandler (row 0)
    const int j0 = C.row0();
    double cur2 = -1.0, last = -1.0;
    for (int i = T.n_lw; i < D; ++i) {
        if (!C.off(i) || j0 < 0) continue;
        const double d2 = C.dist2(j0, i);
        if (cur2 < 0 || d2 < cur2) cur2 = d2;
        const double ld = last_dist[i - T.n_lw];
        if (ld == ld && (last < 0 || ld < last)) last = ld;
    }
    const double current = sqrt(fmax(cur2, 0.0));
    const double munition = (double)m.g[0], reload = (double)fmax(T.cooldown - ((double)w[W_STEP] - (double)S.last[b]), 0.0) / T.cooldown;
    const bool avail = m.g[2] == 1.f;
    double score = (avail || munition == 0.0) ? -current : current * (2 * reload - 1);
    double bonus = 0, penalty = 0;
    if (0.01 < last - current && (avail || munition == 0.0))
        bonus += 10.0 * norm3((double)ag[AG_UB], (double)ag[AG_VB], (double)ag[AG_WB]);
    bonus += 1000.0 * shots;
    penalty += 1000.0 * exploded;
    const int lw_out = C.count_outside_dome(0, T.n_lw);
    if (lw_out > 0) penalty += 1000.0;
    m.reward = score + bonus - penalty;
    int n_armed_lw = 0;
    for (int j = 0; j < T.n_lw; ++j) n_armed_lw += C.live(j) ? 1 : 0;
    m.done = w[W_STEP] > w[W_MAX_STEP];             // compute_termination stages.py:298-344
    m.done |= lw_out > 0;
    m.done |= C.count_outside_dome(T.n_lw, D) > 0;
    m.done |= n_armed_lw < T.n_lw;
    return m;
}
// disarmed munitions reappear at once (stages.py:170-174,370-376); on_step_end: last offsets := current
template <typename R, int FAM, int GS> __device__ __forceinline__ void stage02_on_step_end(EnvCtx<R, FAM, GS>& C, double* last_dist) {
    const TaskParams& T = C.T;
    int32_t* w = C.w;
    const int D = T.D;
    int n_dead = 0;
    for (int i = T.n_lw; i < D; ++i) n_dead += C.live(i) ? 0 : 1;
    if (n_dead > 0) {
        const uint32_t base = (uint32_t)w[W_SPAWN_CTR];
        int k = 0;
        for (int i = T.n_lw; i < D; ++i) {
            if (C.live(i)) continue;
            double p[3];
            C.gen3(base, n_dead, k++, T.respawn_r0, T.respawn_r1, p);
            C.replace(i, p[0], p[1], p[2]);
            C.arm(i);
        }
        w[W_SPAWN_CTR] += 3 * n_dead;
    }
    const int j0 = C.row0();
    const double qnan = __longlong_as_double(0x7ff8000000000000LL);
    for (int i = T.n_lw; i < D; ++i)
        last_dist[i - T.n_lw] = (C.off(i) && j0 >= 0) ? sqrt(C.dist2(j0, i)) : qnan;
}

// ================= level5: Level5C1FusionTask.on_step_middle (level5_c1_fusion_task.py:298-336) =================
template <typename R, int FAM, int GS> __device__ __forceinline__ StepMiddle level5_on_step_middle(EnvCtx<R, FAM, GS>& C, const R* ag, const double* ap) {
    const TaskParams& T = C.T;
    Smem<R>& S = C.S;
    int32_t* w = C.w;
    int32_t* w5 = C.w5;
    const int b = C.b, D = T.D;
    const double apx = ap[0], apy = ap[1], apz = ap[2];
    StepMiddle m;
    const int as = C.agent;
    int agent_shots = 0, ally_shots = 0;
    C.nearest_all();
    for (int j = 0; j < T.n_lw; ++j) {              // process_shoot_range_invaders :399-424
        if (!C.off(j)) continue;
        const int tgt = C.nearest_shoot(j);
        if (tgt < 0) continue;
        if (!(C.gun_available(j) && S.ammo[b + j] > 0)) continue;
        S.ammo[b + j] -= 1; S.last[b + j] = (R)C.gstep();
        const double u = hit_uniform(T.k0, T.k1, C.env_id, (uint32_t)w[W_HIT_CTR]);
        w[W_HIT_CTR] += 1;
        if (u < T.fire_p) { C.disarm(tgt); if (j == as) ++agent_shots; else ++ally_shots; }
    }
    int exploded = 0, agent_suicide = 0, ally_suicide = 0;
    for (int j = 0; j < T.n_lw; ++j) {              // process_explosion_range_invaders :366-397
        if (!C.off(j)) continue;
        const int tgt = C.nearest_expl(j);
        if (tgt < 0) continue;
        C.disarm(j); C.disarm(tgt);
        if (S.ammo[b + j] == 0 && j == as) ++agent_suicide;
        else if (S.ammo[b + j] == 0) ++ally_suicide;
        else ++exploded;
    }
    w[W_AGENT_KILLS] += agent_shots; w[W_ALLIES_KILLS] += ally_shots; w[W_DEADS] += exploded;
    for (int i = T.n_lw; i < D; ++i)                   // process_invaders_in_origin
        if (C.off(i) && sq3(C.pos(i, 0), C.pos(i, 1), C.pos(i, 2)) < 0.2 * 0.2) C.disarm(i);
    if (FAM == FAM_L5_MULTI && T.l5_eval) m.reward = 0.0;                 // "EVALUATION TASK DO NOT USES REWARD" (level5_2bt_evaluation_task.py:418-427)
    else if (T.reward == 2) {
        // Level5FusionTask.compute_reward (level5_fusion_task.py:448-555; allies_dead is never passed)
        double score, bonus = 0, penalty = 0;
        const bool avail = C.gun_available(as);
        const int ammo = S.ammo[b + as];
        const int target = C.ally_target(as);
        double tpx = 0, tpy = 0, tpz = 0;
        if (target >= 0) { tpx = C.pos(target, 0); tpy = C.pos(target, 1); tpz = C.pos(target, 2); }
        const double current = norm3(apx - tpx, apy - tpy, apz - tpz);
        if (avail || ammo == 0) score = -current;
        else {
            score = current;
            if (current < 5.0) penalty += ((5.0 - current) / 5.0) * (0.50 * 1000.0);
        }
        if (!avail && ammo > 0 && (current - C.last_closest()) > 0.01) bonus += 0.10 * 1000.0;
        if (agent_shots > 0) bonus += 1.0 * agent_shots * 1000.0;
        if (ally_shots > 0 || ally_suicide > 0) bonus += 0.5 * (ally_shots + ally_suicide) * 1000.0;
        if (agent_suicide > 0) penalty += 2.0 * agent_suicide * 1000.0;
        if (exploded > 0) penalty += 1000.0 * exploded;
        if (apz < -5.0) penalty += fmin((-5.0 - apz) / 1.0, 1.0) * 1000.0;
        if (C.count_outside_dome(0, T.n_lw) > 0) penalty += 1000.0;
        const double d0 = norm3(apx, apy, apz);
        if (d0 > T.born - 2) penalty += fmin((d0 - (T.born - 2)) * 1.0, 1000.0);
        C.set_last_closest(current);
        m.reward = fmin(fmax(score + bonus - penalty, -3000.0), 3000.0);
    } else {
        // compute_reward :434-484: one-shot last_distance, clipped
        const int target = C.off(as) ? C.nearest_invader(as) : -1;
        double tpx = 0, tpy = 0, tpz = 0;
        if (target >= 0) { tpx = C.pos(target, 0); tpy = C.pos(target, 1); tpz = C.pos(target, 2); }
        const double distance = norm3(apx - tpx, apy - tpy, apz - tpz);
        double last_distance = __longlong_as_double(((long long)w5[W5_LAST_DIST_HI] << 32) | (unsigned int)w5[W5_LAST_DIST_LO]);
        if (last_distance != last_distance) {          // ``hasattr(self, 'last_distance')``: set once per env object
            last_distance = distance;
            const long long bits = __double_as_longlong(distance);
            w5[W5_LAST_DIST_LO] = (int32_t)(bits & 0xffffffffLL); w5[W5_LAST_DIST_HI] = (int32_t)(bits >> 32);
        }
        if (distance < last_distance) m.reward += 10.0 * norm3((double)ag[AG_UB], (double)ag[AG_VB], (double)ag[AG_WB]);
        if (agent_shots > 0) m.reward += 1.0 * agent_shots * 1000.0;
        if (agent_suicide > 0) m.reward -= 2.0 * agent_suicide * 1000.0;
        m.reward = fmin(fmax(m.reward, -3000.0), 3000.0);
    }
    if (agent_shots + ally_shots > 0) w[W_MAX_STEP] += T.step_increment;
    // compute_termination :488-545
    const int lw_out = C.count_outside_dome(0, T.n_lw);
    for (int i = T.n_lw; i < D; ++i) m.lm_alive |= C.live(i);
    for (int j = 0; j < T.n_lw; ++j) m.lw_alive |= C.live(j);
    m.all_over = !m.lm_alive && w[W_ROUND] >= T.max_rounds;
    m.done = C.gstep() > w[W_MAX_STEP];
    m.done |= m.all_over;
    m.done |= lw_out > 0;
    m.done |= C.count_outside_dome(T.n_lw, D) > 0;
    m.done |= !m.lw_alive;
    if (FAM != FAM_L5_MULTI) m.done |= !C.live(as);
    if (!(FAM == FAM_L5_MULTI && T.l5_eval)) m.done |= apz < -5.99;
    C.gun_state(C.agent, m.g);
    return m;
}
// Task.on_step_end :338-350 + advance_round :139-152 (setup_round disarms every munition first: the id clash zeroes the
// guns' step until the next broadcast)
template <typename R, int FAM, int GS> __device__ __forceinline__ void level5_on_step_end(EnvCtx<R, FAM, GS>& C, const StepMiddle& m) {
    const TaskParams& T = C.T;
    Smem<R>& S = C.S;
    int32_t* w = C.w;
    int32_t* w5 = C.w5;
    if (!m.all_over && !m.lm_alive && m.lw_alive) C.advance_round();
    if (T.l5_base) {
        // base env: a dead agent still runs read_data -> six empty spheres; the candidates of
        // get_random_neighborhood are the wingmen with an open buffer in the agent's ring at ITS read_data of
        // the first compute_observation call: the armed ones, the ones that died before this step (their LiDAR
        // broadcasts re-opened it) and, of those that died in this step, the ones in front of the agent
        int cand = 0;
        for (int P = 0; P < T.n_lw; ++P)
            if (C.live(P) || !(S.ev[C.b + P] & EV_WAS_ARMED) || P < C.agent) cand |= 1 << P;
        w5[W5_STACK_MODE] = (C.live(C.agent) ? STACK_BUILD : STACK_EMPTY) | (cand << 8);
        w5[W5_OBS_CALL] += 3;
    } else {
        w5[W5_STACK_MODE] = (FAM == FAM_L5_MULTI || C.live(C.agent)) ? STACK_BUILD : STACK_KEEP;   // a dead agent's flight state keeps its last stack
        w5[W5_OBS_CALL] += 1;
    }
    S.envflag[C.le] |= (w[W_STEP] % RING) << 8;     // ring slot of this step for the feature pass
}
// Level5DumbMultiObs.compute_info (level5_dumb_multiobs.py:112-150): inertial + gun vector of every ARMED wingman, at the
// point between on_step_middle and on_step_end
template <typename R, int FAM, int GS> __device__ __forceinline__ void write_multi_info(const EnvCtx<R, FAM, GS>& C, const StepArgs<R>& A, int env) {
    const TaskParams& T = C.T;
    for (int P = 0; P < T.n_lw; ++P) {
        const bool here = C.live(P);
        A.mo_present[(long long)env * T.n_lw + P] = here ? 1 : 0;
        if (!here) continue;
        const V4<R>* rp = reinterpret_cast<const V4<R>*>(A.p.agent + ((long long)env * T.n_rec + P) * AG_WORDS);
        const V4<R> r0 = ld4(rp), r1 = ld4(rp + 1), r2 = ld4(rp + 2);
        float gp3[3]; C.gun_state(P, gp3);
        float* o = A.mo_inertial + ((long long)env * T.n_lw + P) * 15;
        o[0] = nrm<R>(C.pos(P, 0), C.inv_dome); o[1] = nrm<R>(C.pos(P, 1), C.inv_dome); o[2] = nrm<R>(C.pos(P, 2), C.inv_dome);
        o[3] = nrm<R>(r0.x, INV_SPEED); o[4] = nrm<R>(r0.y, INV_SPEED); o[5] = nrm<R>(r0.z, INV_SPEED);
        o[6] = nrm<R>(r0.w, INV_PI); o[7] = nrm<R>(r1.x, INV_PI); o[8] = nrm<R>(r1.y, INV_PI);
        o[9] = nrm<R>(r1.z, INV_2PI); o[10] = nrm<R>(r1.w, INV_2PI); o[11] = nrm<R>(r2.x, INV_2PI);
        o[12] = gp3[0]; o[13] = gp3[1]; o[14] = gp3[2];
    }
}
// ================= stage03 (level4 tasks, FAM_DRIVEN too): Task.on_step_middle exp02_vFinal_task.py:284-318 =================
template <typename R, int FAM, int GS> __device__ __forceinline__ StepMiddle stage03_on_step_middle(EnvCtx<R, FAM, GS>& C, const StepArgs<R>& A, int env, const R* ag, const double* ap) {
    const TaskParams& T = C.T;
    Smem<R>& S = C.S;
    int32_t* w = C.w;
    const int b = C.b, D = T.D, gl = C.g;
    const double apx = ap[0], apy = ap[1], apz = ap[2];
    StepMiddle m;
    if (T.reward == 1) {                               // update_building_life (exp02_v2_full_task.py)
        int cnt = 0;
        for (int i = T.n_lw + gl; i < D; i += GS)
            if (C.off(i) && sq3(C.pos(i, 0), C.pos(i, 1), C.pos(i, 2)) < 0.2 * 0.2) ++cnt;
        w[W_BUILDING] = max(w[W_BUILDING] - C.gsum(cnt), 0);
    }
    // process_shoot_range_invaders :391-412 -> shoot_by_ids -> Gun.shoot
    int agent_shots = 0, ally_shots = 0;
    C.nearest_all();
    for (int j = 0; j < T.n_lw; ++j) {
        if (!C.off(j)) continue;
        const int tgt = C.nearest_shoot(j);
        if (tgt < 0) continue;
        if (!(C.gun_available(j) && S.ammo[b + j] > 0)) continue;
        { const int am = S.ammo[b + j]; C.gsync(); S.ammo[b + j] = am - 1; }      // every lane of the group stores the same value
        S.last[b + j] = (R)w[W_STEP];
        const double u = hit_uniform(T.k0, T.k1, C.env_id, (uint32_t)w[W_HIT_CTR]);
        w[W_HIT_CTR] += 1;
        if (u < T.fire_p) {
            C.disarm(tgt); if (j == 0) ++agent_shots; else ++ally_shots;
            if (FAM == FAM_DRIVEN) A.p.lw_kills[(long long)env * T.n_lw + j] += 1;       // Evaluation_Task.lw_kills :491-494
        }
    }
    // process_explosion_range_invaders :358-389 (same, now stale, distance matrix)
    int exploded = 0, ally_suicide = 0, agent_suicide = 0;
    for (int j = 0; j < T.n_lw; ++j) {
        if (!C.off(j)) continue;
        const int tgt = C.nearest_expl(j);
        if (tgt < 0) continue;
        C.disarm(j); C.disarm(tgt);
        if (T.reward == 1) ++exploded;
        else if (S.ammo[b + j] == 0 && j == 0) ++agent_suicide;
        else if (S.ammo[b + j] == 0) ++ally_suicide;
        else ++exploded;
    }
    const bool EVAL = FAM == FAM_DRIVEN && T.eval_task;     // Evaluation_Task.on_step_middle evaluation_task.py:383-407
    if (!EVAL) {
        w[W_AGENT_KILLS] += agent_shots; w[W_ALLIES_KILLS] += ally_shots; w[W_DEADS] += exploded;
        C.gsync();
        for (int i = T.n_lw + gl; i < D; i += GS)       // process_invaders_in_origin :656-659
            if (C.off(i) && sq3(C.pos(i, 0), C.pos(i, 1), C.pos(i, 2)) < 0.2 * 0.2) C.disarm(i);
        C.gsync();
    }

    // ---- reward ----
    C.gun_state(C.agent, m.g);
    const int lw_out = C.count_outside_dome(0, T.n_lw);
    if (EVAL) m.reward = 0.0;                        // "Reward will be deactivated" (evaluation_task.py:512-516)
    else if (T.reward == 0) {                        // exp02_vFinal_task.py:422-514
        double bonus = 0, penalty = 0, score;
        const double munition = (double)S.ammo[b] / (double)(T.munition > 0 ? T.munition : 1);
        const double reload = fmax(T.cooldown - ((double)w[W_STEP] - (double)S.last[b]), 0.0) / T.cooldown;
        const bool avail = C.gun_available(0);
        const int target = C.ally_target(0);
        double tpx = 0, tpy = 0, tpz = 0;
        if (target >= 0) { tpx = C.pos(target, 0); tpy = C.pos(target, 1); tpz = C.pos(target, 2); }
        const double current = norm3(apx - tpx, apy - tpy, apz - tpz);
        if (0.01 < C.last_closest() - current && (avail || munition == 0.0))
            bonus += T.vel_bonus * norm3((double)ag[AG_UB], (double)ag[AG_VB], (double)ag[AG_WB]);
        C.set_last_closest(current);
        score = (avail || munition == 0.0) ? -current : current * (2 * reload - 1);
        if (agent_shots > 0 || agent_suicide > 0) bonus += (agent_shots + agent_suicide) * 1000.0;
        if (ally_shots > 0 || ally_suicide > 0) bonus += 0.5 * (ally_shots + ally_suicide) * 1000.0;
        else if (exploded > 0) penalty += 1000.0 * exploded;
        if (apz < -5.0) penalty += (-5.0 - apz) / (-5.0 + 6.0) * 1000.0;
        if (lw_out > 0) penalty += 1000.0;
        const double d0 = norm3(apx, apy, apz);
        if (d0 > T.born - 2) penalty += d0 - T.born - 2;
        m.reward = score + bonus - penalty;
    } else {                                         // exp02_v2_full_task.py compute_reward
        double bonus = 0, penalty = 0;
        const int shots = agent_shots + ally_shots;
        const double kills = (double)(w[W_AGENT_KILLS] + w[W_ALLIES_KILLS]);
        if (shots > 0) bonus += (shots + kills / 10) * 1000.0;
        if (S.ammo[b] == 0 && exploded > 0) bonus += (shots + kills / 10) * 1000.0;
        else if (exploded > 0) penalty += 1000.0 * exploded;
        if (apz < 0.01) penalty += 1000.0;
        if (lw_out > 0) penalty += 1000.0;
        if (w[W_BUILDING] < 1) penalty += 1000.0 * (1 - w[W_BUILDING]);
        const double d0 = norm3(apx, apy, apz);
        if (d0 > T.born) penalty += d0 - T.born;
        m.reward = 0 + bonus - penalty;
    }
    if (agent_shots + ally_shots > 0) w[W_MAX_STEP] += T.step_increment;   // increment_max_step :149-152

    // ---- termination :516-568 ----
    for (int i = T.n_lw + gl; i < D; i += GS) m.lm_alive |= C.live(i);
    m.lm_alive = C.gany(m.lm_alive);
    for (int j = 0; j < T.n_lw; ++j) m.lw_alive |= C.live(j);
    m.all_over = !m.lm_alive && w[W_ROUND] >= T.n_lm;
    m.done = w[W_STEP] > w[W_MAX_STEP] && !(EVAL && !T.time_limited);      // evaluation_task.py:522
    m.done |= m.all_over;
    if (T.reward == 1) m.done |= w[W_BUILDING] <= 0;
    m.done |= lw_out > 0;
    m.done |= C.count_outside_dome(T.n_lw, D) > 0;
    m.done |= !m.lw_alive;
    if (!EVAL) {                                     // a training env stops when its agent dies; the evaluation goes on
        m.done |= !C.live(0);
        m.done |= apz < (T.reward == 1 ? 0.01 : -5.99);
    }
    if (FAM == FAM_DRIVEN && A.lw_info) {            // compute_info (evaluation_task.py:554-574), between middle and end
        for (int j = 0; j < T.n_lw; ++j)
            reinterpret_cast<int4*>(A.lw_info)[(long long)env * T.n_lw + j] =
                make_int4(A.p.lw_kills[(long long)env * T.n_lw + j], C.live(j) ? 1 : 0, S.ammo[b + j], 0);
    }
    return m;
}
// The inertial observation of wingman P right after Env.reset: its new position, zero velocities and attitude, a fresh
// gun.  Wingman C.agent gives the agent's vector; write_multi_reset gives those of the multi-observer rows.
template <typename R, int FAM, int GS> __device__ __forceinline__ void reset_inertial(const EnvCtx<R, FAM, GS>& C, int P, float* o) {
    const int rp = 3 * (C.b + P);
    o[0] = nrm<R>(C.S.newpos[rp], C.inv_dome); o[1] = nrm<R>(C.S.newpos[rp + 1], C.inv_dome); o[2] = nrm<R>(C.S.newpos[rp + 2], C.inv_dome);
    for (int k = 3; k < 12; ++k) o[k] = 0.f;
    float g[3]; C.gun_state(P, g);
    o[12] = g[0]; o[13] = g[1]; o[14] = g[2];
}
// multi-observer reset observation: every wingman re-armed at its new position
template <typename R, int FAM, int GS> __device__ __forceinline__ void write_multi_reset(const EnvCtx<R, FAM, GS>& C, const StepArgs<R>& A, int env) {
    for (int P = 0; P < C.T.n_lw; ++P) {
        A.mo_present[(long long)env * C.T.n_lw + P] = 1;
        reset_inertial(C, P, A.mo_inertial + ((long long)env * C.T.n_lw + P) * 15);
    }
}

// ------------------------------------------------------------------------------------------------
// P4: the LiDAR passes of one warp over its envs [LE_LO, LE_HI) and slots [S_LO, S_HI) of the block.
// ------------------------------------------------------------------------------------------------
// a cell of the agent's sphere given back (LIDARSpec.empty_sphere), and a cell marked by entity d (EntityType value / 5,
// normalised age 1/10: lidar_buffer.py:98-99)
__device__ __forceinline__ void sphere_clear(float* sph, int c, int ch) {
    sph[c] = 1.0f; sph[N_CELLS + c] = 1.0f;
    if (ch == 3) sph[2 * N_CELLS + c] = 1.0f;
}
__device__ __forceinline__ void sphere_mark(float* sph, int c, float rn, bool is_lw, int ch) {
    sph[c] = rn;
    sph[N_CELLS + c] = (float)((is_lw ? 3.0 : 1.0) / 5.0);
    if (ch == 3) sph[2 * N_CELLS + c] = 0.1f;
}
// (cell, r_n) of the entity at imu position e in the frame of the agent at o with the attitude of its record ag.
// F32 (float32 build, fused flavour): float32 projection, exact cell (lidar_cell_fused_f32).  Otherwise the fused flavour
// projects in float64 from the float32 snapshot (perception_snapshot.py:91-110), the classic one in float64.
template <typename R, bool F32> __device__ __forceinline__ void project_agent(const TaskParams& T, const R* o, const R* ag, const R* e, int* cell, double* rn) {
    if (F32 && T.lidar == 0 && sizeof(R) == 4) {
        int c; float r;
        lidar_cell_fused_f32((float)(2 * T.dome), (float)o[0], (float)o[1], (float)o[2],
                             (float)ag[AG_QX], (float)ag[AG_QY], (float)ag[AG_QZ], (float)ag[AG_QW],
                             (float)e[0], (float)e[1], (float)e[2], &c, &r);
        *cell = c; *rn = (double)r;
    } else if (T.lidar == 0) {
        int c; double r;
        lidar_cell_fused(2 * T.dome, (double)(float)o[0], (double)(float)o[1], (double)(float)o[2],
                         (double)(float)ag[AG_QX], (double)(float)ag[AG_QY], (double)(float)ag[AG_QZ], (double)(float)ag[AG_QW],
                         (double)(float)e[0], (double)(float)e[1], (double)(float)e[2], &c, &r);
        *cell = c; *rn = r;
    } else {
        const LidarHit h = lidar_project_one(1, 2 * T.dome, (double)o[0], (double)o[1], (double)o[2],
                                             (double)ag[AG_QX], (double)ag[AG_QY], (double)ag[AG_QZ], (double)ag[AG_QW],
                                             (double)e[0], (double)e[1], (double)e[2]);
        *cell = h.cell; *rn = h.rn;
    }
}

// level5: every armed wingman P runs FusedLIDAR.update_data (level5_c1_fusion_environment.py:25-26); what the agent's
// ring keeps of it -- P's float32 pose and the kept features (r_n, theta, phi float64, type, id) -- goes to ring slot
// step % 10.  stack_kernel assembles the observation from the ring afterwards.
template <typename R> __device__ __forceinline__ void level5_ring_pass(const StepArgs<R>& A, const Smem<R>& S, int env0, int S_LO, int S_HI, int lane) {
    const TaskParams& T = A.t;
    const int D = T.D;
    int* s_list = S.list + S_LO;
    for (int P = 0; P < T.n_lw; ++P) {
        for (int s = S_LO + lane; s < S_HI; s += 32) { S.cell[s] = -1; S.rn[s] = 1.0; }
        int n_proj = 0;
        for (int s = S_LO + lane; s < S_HI + lane; s += 32) {
            bool pred = false;
            if (s < S_HI) {
                const int le = A.env_of(s), d = s - le * D;
                pred = d != P && (S.ev[s] & EV_MID) && (S.ev[le * D + P] & EV_MID) && (S.envflag[le] & EF_LIDAR);
            }
            n_proj = warp_compact(pred, s, s_list, n_proj);
        }
        __syncwarp();
        for (int i = lane; i < n_proj; i += 32) {
            const int s = s_list[i];
            const int le = A.env_of(s), o = le * D + P;
            const R* rec = A.p.agent + ((long long)(env0 + le) * T.n_rec + P) * AG_WORDS;
            const LidarHit h = lidar_project_one(0, 2 * T.dome, (double)(float)S.imu[3 * o], (double)(float)S.imu[3 * o + 1],
                                                 (double)(float)S.imu[3 * o + 2], (double)(float)rec[AG_QX], (double)(float)rec[AG_QY],
                                                 (double)(float)rec[AG_QZ], (double)(float)rec[AG_QW],
                                                 (double)(float)S.imu[3 * s], (double)(float)S.imu[3 * s + 1], (double)(float)S.imu[3 * s + 2]);
            S.cell[s] = h.cell; S.rn[s] = h.rn; S.ang[2 * s] = h.theta; S.ang[2 * s + 1] = h.phi;
        }
        __syncwarp();
        for (int s = S_LO + lane; s < S_HI; s += 32) {
            const int le = A.env_of(s), d = s - le * D, b = le * D;
            if (!(S.envflag[le] & EF_LIDAR) || !(S.ev[b + P] & EV_MID)) continue;
            const long long entry = ((long long)(env0 + le) * T.n_lw + P) * RING + ((S.envflag[le] >> 8) & 15);
            const bool win = lidar_wins(0, d, D, S.cell + b, S.rn + b);
            A.p.ring_meta[entry * D + d] = win ? (S.cell[s] | ((d < T.n_lw ? 3 : 1) << 16)) : -1;
            if (win) {
                double* f = A.p.ring_feat + (entry * D + d) * 3;
                f[0] = S.rn[s]; f[1] = S.ang[2 * s]; f[2] = S.ang[2 * s + 1];
            }
            if (d == P) {
                const R* rec = A.p.agent + ((long long)(env0 + le) * T.n_rec + P) * AG_WORDS;
                float4* pp = reinterpret_cast<float4*>(A.p.ring_pose + entry * 8);
                pp[0] = make_float4((float)S.imu[3 * s], (float)S.imu[3 * s + 1], (float)S.imu[3 * s + 2], (float)rec[AG_QX]);
                pp[1] = make_float4((float)rec[AG_QY], (float)rec[AG_QZ], (float)rec[AG_QW], 0.f);
            }
        }
        __syncwarp();
    }
}

// The agent's sphere (wingman 0 observes).  It lives in the caller's obs_lidar buffer across steps and is maintained
// INCREMENTALLY: the cells held by the previous step's hits (remembered in sphere_desc, parked in S.rn by P0) go back to
// 1.0, then the new hits are written -- bit-identical to rebuilding LIDARSpec.empty_sphere() + add_features, at a few
// dozen bytes per env instead of 4 KB.  When the agent is no longer a publisher nothing is touched: the reference keeps
// the previous sphere (fused_lidar.py:160-166).
// SYNC0 (FAM_DRIVEN, wingman 0 flown by a policy): its FusedLIDAR keeps ONE sphere that the step-start update
// (lw_obs_kernel, dc_buffers.lw_lidar[:,0], SimPtrs::lw_desc) and this end-of-step update both overwrite.  When this
// update is skipped (wingman 0 is no publisher any more) the observation shows that object as the step-start update left
// it.  SYNC0 projects in float64 from the float32 snapshot in both builds.
template <typename R, bool SYNC0> __device__ __forceinline__ void agent_sphere_pass(const StepArgs<R>& A, const Smem<R>& S, int env0, int LE_LO, int LE_HI, int S_LO, int S_HI, int lane) {
    const TaskParams& T = A.t;
    const int D = T.D;
    const long long slot0 = (long long)env0 * D;
    const int ch = T.lidar == 0 ? 3 : 2;
    const int per_env = ch * N_CELLS;
    int* s_list = S.list + S_LO;
    if (A.lidar_ids) {
        int32_t* idp = A.lidar_ids + (long long)(env0 + LE_LO) * N_CELLS;
        for (int i = lane; i < (LE_HI - LE_LO) * N_CELLS; i += 32) idp[i] = -1;   // features = [] when skipped
    }
    // One pass over the warp's slots: a slot whose entity held a cell of the previous sphere gives it back (cell and,
    // without SYNC0, remembered-hit record; SYNC0 gives back the cells of every env), and the entities that can mark a
    // cell now -- alive after the engagement, not the observer, observer still a publisher -- are compacted so that the
    // float64 projection runs on full warps.
    int n_proj = 0;
    for (int s = S_LO + lane; s < S_HI + lane; s += 32) {
        bool pred = false;
        if (s < S_HI) {
            const int le = A.env_of(s), d = s - le * D;
            const bool on = S.envflag[le] & EF_LIDAR;
            const int oc = (int)reinterpret_cast<const long long*>(S.rn)[s];
            if ((on || SYNC0) && oc >= 0) {
                sphere_clear(A.obs_lidar + (long long)(env0 + le) * per_env, oc, ch);
                if (!SYNC0) A.p.sphere_desc[slot0 + s] = make_int2(-1, __float_as_int(1.0f));
            }
            pred = d != 0 && (S.ev[s] & EV_MID) && on;
            S.cell[s] = -1;
        }
        n_proj = warp_compact(pred, s, s_list, n_proj);
    }
    __syncwarp();                                 // un-write before write: two slots of an env may name the same cell
    if (SYNC0) {                                  // the envs without this update show the step-start sphere of wingman 0
        for (int s = S_LO + lane; s < S_HI; s += 32) {
            const int le = A.env_of(s), d = s - le * D;
            if (S.envflag[le] & EF_LIDAR) continue;
            const int2 h = A.p.lw_desc[((long long)(env0 + le) * T.n_lw + 0) * D + d];
            A.p.sphere_desc[slot0 + s] = make_int2(h.x >= 0 ? h.x : -1, h.x >= 0 ? h.y : __float_as_int(1.0f));
            if (h.x >= 0) sphere_mark(A.obs_lidar + (long long)(env0 + le) * per_env, h.x, __int_as_float(h.y), d < T.n_lw, ch);
        }
    }
    DC_STAMP_STEP(6);
    for (int i = lane; i < n_proj; i += 32) {
        const int s = s_list[i];
        const int b = A.env_of(s) * D;
        const R* ag = A.p.agent + (long long)(env0 + A.env_of(s)) * T.n_rec * AG_WORDS;      // record of wingman 0
        project_agent<R, !SYNC0>(T, S.imu + 3 * b, ag, S.imu + 3 * s, S.cell + s, S.rn + s);
    }
    __syncwarp();
    DC_STAMP_STEP(7);
    // winners among the projected entities (full warps): into the sphere, and remembered for the next step's
    // un-write (and for the sparse host transfer)
    for (int i = lane; i < n_proj; i += 32) {
        const int s = s_list[i];
        const int le = A.env_of(s), d = s - le * D, b = le * D;
        if (!lidar_wins(T.lidar, d, D, S.cell + b, S.rn + b)) continue;
        if (SYNC0) S.ev[s] |= EV_LWIN;
        const int c = S.cell[s];
        const float rnf = (float)S.rn[s];
        sphere_mark(A.obs_lidar + (long long)(env0 + le) * per_env, c, rnf, d < T.n_lw, ch);
        if (A.lidar_ids) A.lidar_ids[(long long)(env0 + le) * N_CELLS + c] = d;
        if (!SYNC0) A.p.sphere_desc[slot0 + s] = make_int2(c, __float_as_int(rnf));
    }
    if (SYNC0) {                                  // the record of every slot of an env with this update
        __syncwarp();
        for (int s = S_LO + lane; s < S_HI; s += 32) {
            if (!(S.envflag[A.env_of(s)] & EF_LIDAR)) continue;
            const bool win = S.ev[s] & EV_LWIN;
            A.p.sphere_desc[slot0 + s] = make_int2(win ? S.cell[s] : -1, __float_as_int(win ? (float)S.rn[s] : 1.0f));
        }
    }
}

// MODE_RESET, first use of an env: an empty sphere (level5: stack of spheres) and no remembered hits
template <typename R, int FAM> __device__ __forceinline__ void first_use_sphere(const StepArgs<R>& A, const Smem<R>& S, int env0, int LE_LO, int LE_HI, int lane) {
    const TaskParams& T = A.t;
    const int D = T.D;
    const long long slot0 = (long long)env0 * D;
    const int per_env = (fam_l5(FAM) ? N_STACK * 3 : (T.lidar == 0 ? 3 : 2)) * N_CELLS;
    for (int e = LE_LO; e < LE_HI; ++e) {
        if (!(S.envflag[e] & EF_FIRST)) continue;
        float* sph = A.obs_lidar + (long long)(env0 + e) * per_env;
        for (int f = lane; f < per_env; f += 32) sph[f] = 1.0f;
        if (A.lidar_ids) for (int f = lane; f < N_CELLS; f += 32) A.lidar_ids[(long long)(env0 + e) * N_CELLS + f] = -1;
        for (int f = lane; f < D; f += 32) A.p.sphere_desc[slot0 + (long long)e * D + f] = make_int2(-1, 0);
    }
}

// What P4 projects from, exported per slot by the FAM_RAYCAST instantiation for raycast_sphere_kernel (raycast_env.cuh) into
// StepArgs::ray_snap: the float32 IMU snapshot position and a flag word -- RS_ENTITY: P4 projects this entity into the agent's
// sphere (alive after the engagement, not the agent, the agent still a publisher); RS_UPDATE (slot 0 only): P4 updates the
// env's sphere this step.  Every other instantiation exports nothing.
enum { RS_ENTITY = 1, RS_UPDATE = 2 };

// KFAM: the family (FAM_*), or FAM_RAYCAST -- the stage03 step plus the export above
template <typename R, int MODE, int KFAM, int GS = 1>
__global__ void __launch_bounds__(ENV_THREADS, (sizeof(R) == 4 ? DC_ENV_MIN_BLOCKS : 1)) env_kernel(const StepArgs<R> A) {
    constexpr int FAM = KFAM == FAM_RAYCAST ? FAM_STAGE03 : KFAM;
    static_assert(GS == 1 || FAM == FAM_STAGE03, "lane groups are built for the stage03 family only");
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const TaskParams& T = A.t;
    // Warp-autonomous: warp wi of the block owns the EPW envs [EPW wi, EPW wi + EPW) of the block and their slots
    // [S_LO, S_HI) through every phase, so the phases are separated by __syncwarp() only and the warps of an SM
    // drift apart (one warp's global-load latency hides under another warp's game logic).  A warp's time is the sum
    // of its dependent latencies, not its instruction count: EPW < 32 leaves lanes idle in the per-env pass P3 but
    // shortens the slot passes P0/P5/P4 in proportion, and the SMs have the room for the extra warps.
    const int D = T.D, EPB = A.epb;
    const int tid = threadIdx.x, lane = tid & 31;
    const int env0 = blockIdx.x * EPB;
    const int nenv = min(EPB, T.n_envs - env0);
    const int LE_LO = min((tid >> 5) * A.epw, nenv), LE_HI = min(LE_LO + A.epw, nenv);
    const int S_LO = LE_LO * D, S_HI = LE_HI * D;
    Smem<R> S = carve_smem<R>(smem_raw, EPB * D, EPB, fam_l5(FAM));
    const long long slot0 = (long long)env0 * D;
    const long long stride = (long long)T.n_envs * D;
    // MODE_STEP: dyn_kernel wrote this step's imu into imu[parity^1]; MODE_RESET edits the snapshot
    // the next dyn_kernel will read, imu[parity].
    const int out_par = MODE == MODE_STEP ? (A.parity ^ 1) : A.parity;
    V4<R>* imu_g = A.p.imu[out_par];

    // ---- P0: flag words and imu records of the block's slots ------------------------------------------
    // All loads of four trips are issued before anything is consumed (a warp runs this chain alone: its time is
    // the sum of its dependent latencies); the imu record is loaded whether the slot is armed or not, and the
    // remembered sphere hit that P4 un-writes is fetched here too and parked in S.rn.
    if (MODE == MODE_STEP) asm volatile("griddepcontrol.wait;" ::: "memory");      // dyn_kernel's writes (see launch_step)
    if (MODE == MODE_STEP && LE_LO + lane < LE_HI) {       // what P3 reads first, one lane per env: on its way during P0
        const long long e = env0 + LE_LO + lane;
        asm volatile("prefetch.global.L2 [%0];" :: "l"(A.p.env + e * ENV_WORDS));
        asm volatile("prefetch.global.L2 [%0];" :: "l"(A.p.agent + e * T.n_rec * AG_WORDS));
        if (A.actions) asm volatile("prefetch.global.L2 [%0];" :: "l"(A.actions + e * 4));
    }
    DC_STAMP(0);
    if (MODE == MODE_STEP) DC_TL_BEGIN(A.tl_slot);
    constexpr bool STASH_DESC = MODE == MODE_STEP && !fam_l5(FAM);
    {
        constexpr int U = 4;
        for (int s0 = S_LO + lane; s0 < S_HI; s0 += 32 * U) {
            int fwv[U]; V4<R> qv[U]; long long dv[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int s = s0 + 32 * u;
                const bool ok = s < S_HI;
                fwv[u] = ok ? A.p.flagw[slot0 + s] : 0;
                // Evaluation_Task: the episode goes on after wingman 0 died and the env keeps observing it
                // (EvaluationEnvironment.compute_observation: get_all_pursuers()[0]): its last imu position / last_fired
                // live on in the snapshot buffer of the previous step (P5 carries them forward)
                const bool KEEP0 = FAM == FAM_DRIVEN && MODE == MODE_STEP && T.eval_task && ok && !(fwv[u] & F_ARMED) && s - A.env_of(s) * D == 0;
                qv[u] = ok ? ld4((KEEP0 ? A.p.imu[A.parity] : imu_g) + slot0 + s) : V4<R>{0, 0, 0, 0};
                if (STASH_DESC) dv[u] = ok ? *reinterpret_cast<const long long*>(A.p.sphere_desc + slot0 + s) : -1LL;
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int s = s0 + 32 * u;
                if (s >= S_HI) continue;
                const int fw = fwv[u];
                const bool armed = fw & F_ARMED;
                S.ammo[s] = fw >> F_AMMO_SHIFT;
                V4<R> q = qv[u];
                const bool keep0 = FAM == FAM_DRIVEN && MODE == MODE_STEP && T.eval_task && s - A.env_of(s) * D == 0;
                if (!(armed || keep0 || (MODE == MODE_RESET && (fw & F_OFF)))) q = V4<R>{0, 0, 0, (R)(-T.cooldown)};
                S.imu[3 * s] = q.x; S.imu[3 * s + 1] = q.y; S.imu[3 * s + 2] = q.z; S.last[s] = q.w;
                S.ev[s] = MODE == MODE_STEP ? (armed ? (EV_LIVE | EV_OFF | EV_WAS_ARMED | EV_SNAP) : 0)     // on_middle_step: snapshot := armed set
                                            : ((armed ? (EV_LIVE | EV_WAS_ARMED) : 0) | ((fw & F_OFF) ? EV_OFF : 0) | ((fw & F_SNAP) ? EV_SNAP : 0));
                if (STASH_DESC) reinterpret_cast<long long*>(S.rn)[s] = dv[u];
            }
        }
    }
    if (LE_LO + lane < LE_HI) S.envflag[LE_LO + lane] = 0;
    __syncwarp();

    DC_STAMP(1);
    // ---- P3: per-env game logic, one thread per env (GS > 1: a group of GS lanes per env, see EnvCtx) ----
    const int gl = GS > 1 ? (lane & (GS - 1)) : 0;
    const bool lead = gl == 0;                               // the lane that stores the env's outputs to global memory
    for (int le = LE_LO + lane / GS; le < LE_HI; le += 32 / GS) {
        const int env = env0 + le, b = le * D;
        int32_t w[ENV_WORDS];
        {
            const int4* wp = reinterpret_cast<const int4*>(A.p.env + (long long)env * ENV_WORDS);
#pragma unroll
            for (int k = 0; k < 4; ++k) { int4 t = wp[k]; w[4 * k] = t.x; w[4 * k + 1] = t.y; w[4 * k + 2] = t.z; w[4 * k + 3] = t.w; }
        }
        EnvCtx<R, FAM, GS> C(T, S, b, le, T.env_offset + (uint32_t)env, w);
        if (GS > 1) { C.g = gl; C.gmask = ((1u << GS) - 1u) << (lane & ~(GS - 1)); }
        if (FAM == FAM_DRIVEN) C.kills = A.p.lw_kills + (long long)env * T.n_lw;
        double* lw_init = A.p.lw_init + (long long)env * T.n_lw * 3;
        double* last_dist = A.p.last_dist + (long long)env * T.n_lm;
        if (fam_l5(FAM)) {
            C.w5 = A.p.env5 + (long long)env * ENV5_WORDS;
            C.agent = C.w5[W5_AGENT]; C.gun_step = C.w5[W5_GUN_STEP]; C.registered = C.w5[W5_REGISTERED] != 0;
        }
        float inertial[15];
        float act[4] = {0.f, 0.f, 0.f, 0.f};
        bool write_obs = false;
        if (MODE == MODE_STEP) {
            R ag[AG_WORDS];
            {
                const V4<R>* agp = reinterpret_cast<const V4<R>*>(A.p.agent + ((long long)env * T.n_rec + C.agent) * AG_WORDS);
#pragma unroll
                for (int k = 0; k < 4; ++k) { V4<R> t = ld4(agp + k); ag[4 * k] = t.x; ag[4 * k + 1] = t.y; ag[4 * k + 2] = t.z; ag[4 * k + 3] = t.w; }
            }
            if (!(FAM == FAM_DRIVEN && T.eval_task)) {              // EvaluationEnvironment.last_action is never set: zeros
                const float4 a4 = reinterpret_cast<const float4*>(A.actions)[env];
                act[0] = a4.x; act[1] = a4.y; act[2] = a4.z; act[3] = a4.w;
            }
            w[W_STEP] += 1; w[W_PHYS_CTR] += T.substeps; w[W_EP_STEPS] += 1;
            C.broadcast_step();                            // advance_step_counter -> AGENT_STEP_BROADCAST
            const double ap[3] = {C.pos(C.agent, 0), C.pos(C.agent, 1), C.pos(C.agent, 2)};
            StepMiddle m;
            if constexpr (FAM == FAM_STAGE01) m = stage01_on_step_middle(C, ag, ap);
            else if constexpr (FAM == FAM_STAGE02) m = stage02_on_step_middle(C, ag, last_dist);
            else if constexpr (fam_l5(FAM)) m = level5_on_step_middle(C, ag, ap);
            else m = stage03_on_step_middle(C, A, env, ag, ap);

            w[W_EP_RETURN] = __float_as_int(__int_as_float(w[W_EP_RETURN]) + (float)m.reward);
            if (lead) {
                A.reward[env] = (float)m.reward;
                A.done[env] = m.done ? 1 : 0;
                int32_t* info = A.info + (long long)env * INFO_WORDS;
                reinterpret_cast<int4*>(info)[0] = make_int4(w[W_AGENT_KILLS], w[W_ALLIES_KILLS], w[W_DEADS], w[W_ROUND]);
                reinterpret_cast<int4*>(info)[1] = make_int4(w[W_BUILDING], w[W_STEP], w[W_MAX_STEP], w[W_EP_STEPS]);
            }

            // ---- observation vector: normalize_inertial_data + gun_state ----
            inertial[0] = nrm<R>(ap[0], C.inv_dome); inertial[1] = nrm<R>(ap[1], C.inv_dome); inertial[2] = nrm<R>(ap[2], C.inv_dome);
            inertial[3] = nrm<R>(ag[AG_UB], INV_SPEED); inertial[4] = nrm<R>(ag[AG_VB], INV_SPEED); inertial[5] = nrm<R>(ag[AG_WB], INV_SPEED);
            inertial[6] = nrm<R>(ag[AG_ROLL], INV_PI); inertial[7] = nrm<R>(ag[AG_PITCH], INV_PI); inertial[8] = nrm<R>(ag[AG_YAW], INV_PI);
            inertial[9] = nrm<R>(ag[AG_P], INV_2PI); inertial[10] = nrm<R>(ag[AG_Q], INV_2PI); inertial[11] = nrm<R>(ag[AG_R], INV_2PI);
            inertial[12] = m.g[0]; inertial[13] = m.g[1]; inertial[14] = m.g[2];
            write_obs = true;
            if (FAM == FAM_L5_MULTI && !T.l5_eval) write_multi_info(C, A, env);

            // LiDAR is rebuilt only while the agent is still a publisher (fused_lidar.py:160-166)
            C.gsync();
            for (int k = gl; k < D; k += GS) if (S.ev[b + k] & EV_LIVE) S.ev[b + k] |= EV_MID;
            C.gsync();
            if (C.live(C.agent)) S.envflag[le] |= EF_LIDAR;

            if constexpr (FAM == FAM_STAGE01) stage01_on_step_end(C, m, ap);
            else if constexpr (FAM == FAM_STAGE02) stage02_on_step_end(C, last_dist);
            else if constexpr (fam_l5(FAM)) level5_on_step_end(C, m);
            else if (!m.all_over && !m.lm_alive && m.lw_alive) C.advance_round();    // Task.on_step_end :320-332
            // ---- VecEnv auto-reset (SB3 DummyVecEnv.step_wait semantics) ----
            if (m.done && T.auto_reset) {
                if (A.term_inertial && lead) for (int k = 0; k < 15; ++k) A.term_inertial[(long long)env * 15 + k] = inertial[k];
                if (A.term_last_action && lead) reinterpret_cast<float4*>(A.term_last_action)[env] = make_float4(act[0], act[1], act[2], act[3]);
                if (A.stats && lead) {
                    atomicAdd(A.stats + 0, 1.0); atomicAdd(A.stats + 1, (double)__int_as_float(w[W_EP_RETURN]));
                    atomicAdd(A.stats + 2, (double)w[W_EP_STEPS]); atomicAdd(A.stats + 3, (double)w[W_AGENT_KILLS]);
                    atomicAdd(A.stats + 4, (double)w[W_ALLIES_KILLS]); atomicAdd(A.stats + 5, (double)w[W_DEADS]);
                    atomicAdd(A.stats + 6, (double)w[W_ROUND]);
                }
                C.reset_task(lw_init, last_dist);
                if (fam_l5(FAM)) S.envflag[le] &= ~EF_LIDAR;
                // level5 C1 reports agent.last_action, the command the drone keeps across the reset (quadcopter.py:415-419);
                // the base level5 env reports its own last_action, zeroed by init_globals (level5_envrionment.py:153-155)
                if (!fam_l5(FAM) || T.l5_base) act[0] = act[1] = act[2] = act[3] = 0.f;
                reset_inertial(C, C.agent, inertial);
                if (FAM == FAM_L5_MULTI && !T.l5_eval) write_multi_reset(C, A, env);
            }
        } else {
            // ---- MODE_RESET: Env.__init__ on first use, then Env.reset for the masked envs ----
            const bool masked = A.reset_mask == nullptr || A.reset_mask[env] != 0;
            const bool first = w[W_INIT] == 0;
            if (first) {
                C.init_task(lw_init, last_dist);
                S.envflag[le] |= EF_FIRST;                  // first use: start from an empty sphere
            }
            if (fam_l5(FAM)) C.w5[W5_STACK_MODE] = STACK_KEEP;
            if (masked || first) {
                C.reset_task(lw_init, last_dist);
                reset_inertial(C, C.agent, inertial);
                write_obs = true;
                if (FAM == FAM_L5_MULTI && !T.l5_eval) write_multi_reset(C, A, env);
            }
        }
        if (write_obs && lead) {
            float* oi = A.obs_inertial + (long long)env * 15;
            for (int k = 0; k < 15; ++k) oi[k] = inertial[k];
            if (!(MODE == MODE_RESET && fam_l5(FAM) && !T.l5_base && !(S.envflag[le] & EF_FIRST)))      // level5 C1 reset keeps agent.last_action
                reinterpret_cast<float4*>(A.obs_last_action)[env] = make_float4(act[0], act[1], act[2], act[3]);
        }
        if (fam_l5(FAM)) { C.w5[W5_AGENT] = C.agent; C.w5[W5_GUN_STEP] = C.gun_step; C.w5[W5_REGISTERED] = C.registered ? 1 : 0; }
        int4* wp = reinterpret_cast<int4*>(A.p.env + (long long)env * ENV_WORDS);
#pragma unroll
        for (int k = 0; k < 4; ++k) if (lead) wp[k] = make_int4(w[4 * k], w[4 * k + 1], w[4 * k + 2], w[4 * k + 3]);
    }
    __syncwarp();

    DC_STAMP(2);
    // ---- spawn pass: the munition waves the env pass asked for, one lane per munition; and the work list of the next
    // step (the armed flags are final after P3): warp-local compaction in slot order, then ONE atomic per warp reserves the
    // range -- issued here so that its round trip runs under P5's stores, which do not need the answer.
    int32_t* items_out = A.p.items[out_par];
    int32_t* count_out = A.p.count + out_par;
    int* s_list = S.list + S_LO;                            // the warp's private list (capacity: its own slots)
    int n_before = 0;
    for (int s = S_LO + lane; s < S_HI + lane; s += 32) {    // every lane runs every trip (ballots inside)
        bool live = false;
        if (s < S_HI) {
            const int ev = S.ev[s];
            live = ev & EV_LIVE;
            if (fam_waves(FAM) && (ev & EV_SPAWNJOB)) {
                const int* jp = reinterpret_cast<const int*>(S.newpos + 3 * s);
                const uint32_t base = (uint32_t)jp[0];
                const int n = jp[1], i = jp[2];
                double p[3];
                spawn_point(T, T.env_offset + (uint32_t)(env0 + A.env_of(s)), base, n, i, T.born, p);
                S.newpos[3 * s] = (R)p[0]; S.newpos[3 * s + 1] = (R)p[1]; S.newpos[3 * s + 2] = (R)p[2];
            }
        }
        n_before = warp_compact(live, (int)(slot0 + s), s_list, n_before);
    }
    int gbase = 0;
    if (lane == 0 && n_before > 0) gbase = atomicAdd(count_out, n_before);
    __syncwarp();

    DC_STAMP(3);
    // ---- P5: events -> state (plain stores, nothing is re-read) + the next step's work list -----------
    // In MODE_STEP the next dyn_kernel reads imu[parity^1] and items[parity^1]; in MODE_RESET it reads
    // imu[parity] / items[parity], whose count the host zeroed before this launch.
    for (int s = S_LO + lane; s < S_HI; s += 32) {
        {
            const int le = A.env_of(s);
            const int ev = S.ev[s];
            const bool live = ev & EV_LIVE;
            V4<R>* gp = A.p.state + slot0 + s;
            if (ev & EV_ZEROED) {             // disarm: resetBaseVelocity(0), motors.reset()
                st4(gp + 2 * stride, V4<R>{0, 0, 0, 0}); st4(gp + 3 * stride, V4<R>{0, 0, 0, 0}); st4(gp + 4 * stride, V4<R>{0, 0, 0, 0});
            }
            R ix = S.imu[3 * s], iy = S.imu[3 * s + 1], iz = S.imu[3 * s + 2];
            if (ev & EV_REPLACED) {           // replace: teleport, identity attitude, zero velocity, new formation point
                const R px = S.newpos[3 * s], py = S.newpos[3 * s + 1], pz = S.newpos[3 * s + 2];
                st4(gp, V4<R>{px, py, pz, 0});
                st4(gp + stride, V4<R>{0, 0, 0, 1});
                st4(gp + 2 * stride, V4<R>{0, 0, 0, 0}); st4(gp + 3 * stride, V4<R>{0, 0, 0, 0});
                st4(gp + 12 * stride, V4<R>{px, py, pz, 0});
                if (live) { ix = px; iy = py; iz = pz; }          // update_imu of replace()/arm()
            }
            const int nf = (live ? F_ARMED : 0) | ((ev & EV_OFF) ? F_OFF : 0) | ((ev & EV_SNAP) ? F_SNAP : 0) | ((ev & EV_PENDING) ? F_PENDING : 0) | ((ev & EV_PENDING2) ? F_PENDING2 : 0) |
                           (S.ammo[s] << F_AMMO_SHIFT);
            A.p.flagw[slot0 + s] = nf;
            if (S.envflag[le] & EF_NAV_RESET) A.p.nav[slot0 + s] = NAV_WAIT;
            // imu position | last_fired of every drone that is in the snapshot or alive
            if ((ev & (EV_WAS_ARMED | EV_REARMED | EV_OFF)) || live || (FAM == FAM_DRIVEN && T.eval_task && s - le * D == 0))
                st4(imu_g + slot0 + s, V4<R>{ix, iy, iz, S.last[s]});
        }
    }
    gbase = __shfl_sync(0xffffffffu, gbase, 0);               // the reserved range: a coalesced copy of the warp's list
    for (int i = lane; i < n_before; i += 32) items_out[gbase + i] = s_list[i];
    __syncwarp();                                         // the list is reused by P4

    DC_STAMP(4);
    if (MODE == MODE_STEP) asm volatile("griddepcontrol.launch_dependents;");     // the next step's dyn_kernel waits for the whole grid
    if constexpr (KFAM == FAM_RAYCAST) {
        for (int s = S_LO + lane; s < S_HI; s += 32) {
            const int le = A.env_of(s), d = s - le * D;
            const bool on = MODE == MODE_STEP && (S.envflag[le] & EF_LIDAR);
            const int f = d == 0 ? (on ? RS_UPDATE : 0) : ((on && (S.ev[s] & EV_MID)) ? RS_ENTITY : 0);
            A.ray_snap[slot0 + s] = make_float4((float)S.imu[3 * s], (float)S.imu[3 * s + 1], (float)S.imu[3 * s + 2], __int_as_float(f));
        }
    }
    // ---- P4: LiDAR over the entities alive after engagement --------
    if (MODE == MODE_STEP && fam_l5(FAM)) {
        level5_ring_pass(A, S, env0, S_LO, S_HI, lane);
    } else if (MODE == MODE_STEP) {
        if (FAM == FAM_DRIVEN && A.lw_lidar && (T.lw_driver[0] == DRV_NN || T.lw_driver[0] == DRV_NN_ALLY))
            agent_sphere_pass<R, true>(A, S, env0, LE_LO, LE_HI, S_LO, S_HI, lane);
        else
            agent_sphere_pass<R, false>(A, S, env0, LE_LO, LE_HI, S_LO, S_HI, lane);
        DC_STAMP(5);
        DC_TL_END(A.tl_slot);
    } else {
        first_use_sphere<R, FAM>(A, S, env0, LE_LO, LE_HI, lane);
    }
}

// ================================================================================================
// parity-harness kernels: canonical state layout <-> internal arrays, work-list rebuild
// ================================================================================================
// canonical [13][E*D] quads: 0 pos|flag word (armed, snapshot, nav<<2, ammo<<8), 1..10 as stored,
// 11 imu_pos|last_fired, 12 formation
template <typename R>
__global__ void pack_state_kernel(SimPtrs<R> p, int parity, long long n, V4<R>* out) {
    const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    for (int q = 0; q < STATE_QUADS; ++q) {
        V4<R> v = ld4(p.state + q * n + s);
        if (q == 0) v.w = (R)((p.flagw[s] & 3) | ((int)p.nav[s] << 2) | ((p.flagw[s] >> F_AMMO_SHIFT) << 8));
        if (q == 11) v = ld4(p.imu[parity] + s);
        st4(out + q * n + s, v);
    }
}

template <typename R>
__global__ void unpack_state_kernel(SimPtrs<R> p, int parity, long long n, const V4<R>* in) {
    const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    for (int q = 0; q < STATE_QUADS; ++q) {
        V4<R> v = ld4(in + q * n + s);
        if (q == 0) {
            const int fw = (int)v.w;
            p.flagw[s] = (fw & 3) | ((fw >> 8) << F_AMMO_SHIFT);
            p.nav[s] = (unsigned char)((fw >> 2) & 3);
            v.w = 0;
        }
        if (q == 11) { st4(p.imu[parity] + s, v); st4(p.imu[parity ^ 1] + s, v); }
        st4(p.state + q * n + s, v);
    }
}

__global__ void build_list_kernel(const int32_t* flagw, long long n, int32_t* items, int32_t* count) {
    const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = s < n && (flagw[s] & F_ARMED);
    const unsigned m = __ballot_sync(0xffffffffu, live);
    const int lane = threadIdx.x & 31;
    int wbase = 0;
    if (lane == 0 && m) wbase = atomicAdd(count, __popc(m));
    wbase = __shfl_sync(0xffffffffu, wbase, 0);
    if (live) items[wbase + __popc(m & ((1u << lane) - 1))] = (int)s;
}

}  // namespace dc

// dronechase_b200 -- observations of the wingmen that are flown by policies INSIDE the task (stage03 family FAM_DRIVEN).
//
//   Evaluation_Task.compute_lw_observation   evaluation_task.py:283-312   (drive_lw :257-277, drivers of type "nn")
//   Exp05_vFinal_Task.compute_lw_observation exp05_vFinal_task.py:265-296 (drive_lw_rl_agent :252-260)
//
// Both run at on_step_start: pursuer.update_lidar() (FusedLIDAR.update_data, fused_lidar.py:143-217) on the rings as the
// previous step's on_step_end / the reset left them, then normalize_inertial_data + gun_state, then the task's shared
// last_action (host side).  lw_obs_kernel is that phase for the whole batch: one warp per (env, policy-driven wingman),
// launched by dc_lw_observe before the policies run.  A publisher is visible iff it carries F_SNAP (stage03.cuh): armed at
// the last step broadcast, not disarmed or re-armed since -- so a wave set-up removes every munition from the sphere and a
// reset leaves the previous sphere in place (own snapshot missing: update_data returns early, :160-166).  The snapshot
// positions are the imu positions of the last step (imu[parity]), the observer's quaternion its imu record.
#pragma once
#include "stage03.cuh"

namespace dc {

constexpr int LWOBS_WARPS = 4;
constexpr int LWOBS_MAX_D = 256;
constexpr int LW_DESC_UNUSED = (int)0xFEFEFEFE;      // dc_create fills lw_desc with 0xFE bytes: "lw_lidar row never written"

template <typename R>
__global__ void __launch_bounds__(LWOBS_WARPS * 32) lw_obs_kernel(const StepArgs<R> A) {
    __shared__ int s_cell[LWOBS_WARPS][LWOBS_MAX_D];
    __shared__ double s_rn[LWOBS_WARPS][LWOBS_MAX_D];
    const TaskParams& T = A.t;
    const int D = T.D, L = T.n_lw;
    const int wi = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long job = (long long)blockIdx.x * LWOBS_WARPS + wi;          // (env, wingman)
    if (job >= (long long)T.n_envs * L) return;
    const int env = (int)(job / L), P = (int)(job - (long long)env * L);
    const int drv = T.lw_driver[P];
    if (drv != DRV_NN && drv != DRV_NN_ALLY) return;
    const long long b = (long long)env * D;
    const V4<R>* snap = A.p.imu[A.parity];                                   // imu position | last_fired of the last step
    const int fwP = A.p.flagw[b + P];
    const bool armed = fwP & F_ARMED;
    bool present = armed;
    if (drv == DRV_NN_ALLY) {                                                // get_armed_pursuers()[1:]
        bool before = false;
        for (int j = 0; j < P; ++j) before |= (A.p.flagw[b + j] & F_ARMED) != 0;
        present = armed && before;
    }
    const int per = 3 * N_CELLS;
    float* sph = A.lw_lidar + ((long long)env * L + P) * per;
    int2* desc = A.p.lw_desc + ((long long)env * L + P) * D;
    int* cells = s_cell[wi];
    double* rns = s_rn[wi];
    // ---- first use of this row: an empty sphere ----
    if (desc[0].x == LW_DESC_UNUSED) {
        for (int f = lane; f < per; f += 32) sph[f] = 1.0f;
        for (int d = lane; d < D; d += 32) desc[d] = make_int2(-1, __float_as_int(1.0f));
        __syncwarp();
    }
    const V4<R> own = ld4(snap + b + P);
    const R* rec = A.p.agent + ((long long)env * T.n_rec + P) * AG_WORDS;
    if (lane == 0) {
        A.lw_present[(long long)env * L + P] = present ? 1 : 0;
        if (armed) {
            // normalize_inertial_data (normalization.py:6-110) + Gun.get_state (gun.py:101-113) of wingman P
            auto nrm = [](double v, double inv_scale) { return (float)fmin(fmax(v * inv_scale, -1.0), 1.0); };
            const double inv_dome = 1.0 / T.dome, i_speed = 1.0 / (1 * 10 * (1000.0 / 3600.0));
            const double i_pi = 1.0 / 3.141592653589793, i_2pi = 1.0 / (2 * 3.141592653589793);
            float* o = A.lw_inertial + ((long long)env * L + P) * 15;
            o[0] = nrm(own.x, inv_dome); o[1] = nrm(own.y, inv_dome); o[2] = nrm(own.z, inv_dome);
            if (fwP & F_SNAP) {
                o[3] = nrm(rec[AG_UB], i_speed); o[4] = nrm(rec[AG_VB], i_speed); o[5] = nrm(rec[AG_WB], i_speed);
                o[6] = nrm(rec[AG_ROLL], i_pi); o[7] = nrm(rec[AG_PITCH], i_pi); o[8] = nrm(rec[AG_YAW], i_pi);
                o[9] = nrm(rec[AG_P], i_2pi); o[10] = nrm(rec[AG_Q], i_2pi); o[11] = nrm(rec[AG_R], i_2pi);
            } else {                                      // re-armed at a reset: replace() + arm() -> update_imu at rest
                for (int k = 3; k < 12; ++k) o[k] = 0.f;
            }
            const int ammo = fwP >> F_AMMO_SHIFT;
            const double gstep = (double)A.p.env[(long long)env * ENV_WORDS + W_STEP];
            const double wait = fmax(T.cooldown - (gstep - (double)own.w), 0.0);
            o[12] = (float)((double)ammo / (double)(T.munition > 0 ? T.munition : 1));
            o[13] = (float)(wait / T.cooldown);
            o[14] = (ammo <= 0 || T.cooldown <= gstep - (double)own.w) ? 1.f : 0.f;
        }
    }
    if (!present) return;                                                     // not served: its lidar is not updated
    if (!(fwP & F_SNAP)) {
        // own snapshot missing -> the sphere object keeps its content.  Wingman 0's object is also what the env's
        // compute_observation updates at the end of every step: bring the row to that state (obs_lidar / sphere_desc)
        if (P == 0) {
            for (int d = lane; d < D; d += 32) { const int c = desc[d].x; if (c >= 0) { sph[c] = 1.0f; sph[N_CELLS + c] = 1.0f; sph[2 * N_CELLS + c] = 1.0f; } }
            __syncwarp();
            for (int d = lane; d < D; d += 32) {
                const int2 h = A.p.sphere_desc[b + d];
                desc[d] = h;
                if (h.x < 0) continue;
                sph[h.x] = __int_as_float(h.y); sph[N_CELLS + h.x] = (float)((d < L ? 3.0 : 1.0) / 5.0); sph[2 * N_CELLS + h.x] = 0.1f;
            }
        }
        return;
    }
    // ---- FusedLIDAR.update_data of wingman P over the publishers with a slot-1 snapshot ----
    for (int d = lane; d < D; d += 32) {
        int c = -1; double rn = 1.0;
        if (d != P && (A.p.flagw[b + d] & F_SNAP)) {
            const V4<R> q = ld4(snap + b + d);
            lidar_cell_fused(2 * T.dome, (double)(float)own.x, (double)(float)own.y, (double)(float)own.z,
                             (double)(float)rec[AG_QX], (double)(float)rec[AG_QY], (double)(float)rec[AG_QZ], (double)(float)rec[AG_QW],
                             (double)(float)q.x, (double)(float)q.y, (double)(float)q.z, &c, &rn);
        }
        cells[d] = c; rns[d] = rn;
        const int oc = desc[d].x;                         // un-write what the row shows
        if (oc >= 0) { sph[oc] = 1.0f; sph[N_CELLS + oc] = 1.0f; sph[2 * N_CELLS + oc] = 1.0f; }
    }
    __syncwarp();
    for (int d = lane; d < D; d += 32) {
        const bool win = lidar_wins(0, d, D, cells, rns);
        desc[d] = make_int2(win ? cells[d] : -1, __float_as_int(win ? (float)rns[d] : 1.0f));
        if (!win) continue;
        const int c = cells[d];
        sph[c] = (float)rns[d]; sph[N_CELLS + c] = (float)((d < L ? 3.0 : 1.0) / 5.0); sph[2 * N_CELLS + c] = 0.1f;
    }
}

}  // namespace dc

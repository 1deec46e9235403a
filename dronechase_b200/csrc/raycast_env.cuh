// dronechase_b200 -- the agent's sphere as a ray-cast LiDAR inside a stage03 env (dc_config.lidar = DC_LIDAR_RAYCAST).
//
// An opt-in sensor model: the reference only projects entity centres (lidar.cuh).  raycast_sphere_kernel runs after
// env_kernel<FAM_RAYCAST> of every step and reset and rebuilds the agent's (3,13,26) sphere of each env whose sphere env_kernel's P4
// updated (RS_UPDATE), from the snapshot P4 projected (RS_ENTITY entities, their float32 IMU positions, the agent's record):
//   * every entity claims the cell of its centre at its centre distance, with P4's own projection (project_agent: the float32
//     path of the product build, the float64 one of the verification build);
//   * the ray through the centre of every cell (LidarMath.radian_from_index, rotated body -> world) is tested against the
//     bounding sphere of every entity -- radius ray_r[0] for a wingman, ray_r[1] for a munition -- but only over the
//     entity's angular footprint, the cells whose centre ray can hit it; an observer inside (or on) a sphere sees it at
//     distance 0 in every cell; a radius of 0 casts no ray;
//   * a cell holds the entity with the smaller of its two values, the winner picked in slot order with P4's rule
//     (lidar_wins: strict '<' of the float64 value against the float32 value held) -- nearest first, P4's tie rule after.
// With both radii 0 only the centre claims remain and the sphere, the ids included, is P4's bit for bit.  The whole sphere
// is rewritten, so the incremental state P4 keeps for its own flavour has no influence on what the agent sees.
#pragma once
#include "stage03.cuh"

namespace dc {

constexpr int RAY_ENV_WARPS = 4;      // one env per warp at a time

template <typename R> struct RaySphereArgs {
    TaskParams t;
    const R* agent;              // SimPtrs::agent: the agent's IMU record (attitude quaternion), [E][AG_WORDS]
    const float4* snap;          // env_kernel<FAM_RAYCAST>'s export (StepArgs::ray_snap), [E*D]
    float* obs_lidar;            // [E][3][13][26]
    int32_t* lidar_ids;          // optional [E][13][26]
    float ray_r[2];              // bounding radius of a wingman / of a munition (metres)
};

// per entity of the env a warp works on: centre claim, body-frame offset and the footprint box
template <typename R> struct RayEnt {
    R bx, by, bz;                // offset of the entity in the frame of the agent's rotation matrix: R(q)^T (e - o)
    R rel2;                      // |e - o|^2 (world frame)
    R r2;                        // bounding radius squared
    double rn;                   // centre claim: r_n as P4 computes it
    int cell;                    // centre claim: cell as P4 computes it
    int box;                     // ti0 | nti << 8 | pj0 << 16 | npj << 24 of the cells whose centre ray can hit; 0: none
};

// Footprint of a bounding sphere seen from outside: the rows of cell centres theta_c = (i + 1/2) pi / 13 within alpha + eps
// of the entity's polar angle, and the columns phi_c = -pi + (j + 1/2) 2 pi / 26 within the longitude half-width
// asin(sin(alpha + eps) / sin(theta_e)) + eps of the cap (every column when the widened cap reaches a pole).  eps = 2e-3 rad
// covers the float32 angles (~1e-6 rad) and a quaternion norm off 1 by float32 rounding; it only adds cells to test.
__device__ __forceinline__ int ray_box(float bx, float by, float bz, float dist, float r) {
    const float PI = 3.14159265358979f, EPS = 2e-3f, K = 4.1380285203892786f;       // 13 / pi = 26 / (2 pi)
    // approximate divisions (2 ulp) and sines, so that no slow-path call raises the kernel's register pressure: their
    // errors stay far inside EPS, and the longitude ratio below is bounded from above
    const float a = asinf(fminf(__fdividef(r, dist), 1.0f)) + EPS;
    const float th = acosf(fminf(fmaxf(__fdividef(bz, dist), -1.0f), 1.0f)), ph = atan2f(by, bx);
    const int i0 = max(0, (int)ceilf((th - a) * K - 0.5f)), i1 = min(N_THETA - 1, (int)floorf((th + a) * K - 0.5f));
    if (i1 < i0) return 0;
    int j0 = 0, nj = N_PHI;
    if (th - a > 0.0f && th + a < PI) {
        // an upper bound of sin(a) / sin(th): __sinf is within 1e-6 absolute, and sin(th) > sin(EPS) = 2e-3 here
        const float s = __fdividef(__sinf(a) + 1e-6f, __sinf(th) - 1e-6f);
        if (s < 1.0f) {
            const float w = asinf(s) + EPS;
            const int lo = (int)ceilf((ph - w + PI) * K - 0.5f), hi = (int)floorf((ph + w + PI) * K - 0.5f);
            if (hi < lo) return 0;
            if (hi - lo + 1 < N_PHI) { j0 = ((lo % N_PHI) + N_PHI) % N_PHI; nj = hi - lo + 1; }
        }
    }
    return i0 | ((i1 - i0 + 1) << 8) | (j0 << 16) | (nj << 24);
}

// body-frame unit vector of the centre ray of cell (ti, pj): LidarMath.spherical_to_cartesian of radian_from_index
__device__ __forceinline__ void cell_ray(int ti, int pj, float* x, float* y, float* z) {
    float st, ct, sp, cp;
    sincospif((ti + 0.5f) / N_THETA, &st, &ct);
    sincospif(-1.0f + (pj + 0.5f) / (N_PHI / 2), &sp, &cp);
    *x = st * cp; *y = st * sp; *z = ct;
}
__device__ __forceinline__ void cell_ray(int ti, int pj, double* x, double* y, double* z) {
    double st, ct, sp, cp;
    sincospi((ti + 0.5) / N_THETA, &st, &ct);
    sincospi(-1.0 + (pj + 0.5) / (N_PHI / 2), &sp, &cp);
    *x = st * cp; *y = st * sp; *z = ct;
}

// value of entity E in cell (ti, pj): normalised distance of the first hit of the cell's centre ray, 2 when it misses
template <typename R> __device__ __forceinline__ R ray_value(const RayEnt<R>& E, int ti, int pj, R inv_range) {
    if (E.rel2 <= E.r2) return R(0);                      // the observer is inside (or on) the sphere
    R x, y, z;
    cell_ray(ti, pj, &x, &y, &z);
    const R tca = E.bx * x + E.by * y + E.bz * z;
    if (!(tca > R(0))) return R(2);
    // squared miss distance from the miss vector: |e - o|^2 - tca^2 would cancel catastrophically in float32 (far entities)
    const R mx = E.bx - tca * x, my = E.by - tca * y, mz = E.bz - tca * z;
    const R d2 = mx * mx + my * my + mz * mz;
    if (!(d2 <= E.r2)) return R(2);
    const R t = (tca - sqrt(E.r2 - d2)) * inv_range;
    return t < R(0) ? R(0) : (t > R(1) ? R(1) : t);
}

// P4's winner rule (lidar_wins) for one more candidate of cell c
__device__ __forceinline__ void ray_offer(float* cur, int* win, int c, double v, int k) {
    if (v < (double)cur[c]) { cur[c] = (float)v; win[c] = k; }
}

template <typename R>
__global__ void __launch_bounds__(RAY_ENV_WARPS * 32) raycast_sphere_kernel(const RaySphereArgs<R> A) {
    asm volatile("griddepcontrol.wait;" ::: "memory");  // env_kernel's export (launched with PDL after it)
    extern __shared__ __align__(16) unsigned char ray_smem[];
    const TaskParams& T = A.t;
    const int D = T.D, lane = threadIdx.x & 31, wi = threadIdx.x >> 5;
    float* cur = reinterpret_cast<float*>(ray_smem) + wi * N_CELLS;
    int* win = reinterpret_cast<int*>(ray_smem + RAY_ENV_WARPS * N_CELLS * 4) + wi * N_CELLS;
    RayEnt<R>* ent = reinterpret_cast<RayEnt<R>*>(ray_smem + RAY_ENV_WARPS * N_CELLS * 8) + wi * D;
    const R inv_range = R(1) / (R)(2 * T.dome);          // P4's sphere radius: twice the dome
    for (int env = blockIdx.x * RAY_ENV_WARPS + wi; env < T.n_envs; env += gridDim.x * RAY_ENV_WARPS) {
        const float4* sn = A.snap + (long long)env * D;
        const float4 o4 = sn[0];
        if (!(__float_as_int(o4.w) & RS_UPDATE)) continue;          // P4 kept this env's sphere: so do we
        const R o[3] = {(R)o4.x, (R)o4.y, (R)o4.z};
        const R* ag = A.agent + (long long)env * AG_WORDS;
        const R qx = (R)(float)ag[AG_QX], qy = (R)(float)ag[AG_QY], qz = (R)(float)ag[AG_QZ], qw = (R)(float)ag[AG_QW];
        // R(q) as p.getMatrixFromQuaternion lists it (oracle dynamics.rot_from_quat); the offsets are taken through its transpose
        const R m00 = 1 - 2 * (qy * qy + qz * qz), m01 = 2 * (qx * qy - qw * qz), m02 = 2 * (qx * qz + qw * qy);
        const R m10 = 2 * (qx * qy + qw * qz), m11 = 1 - 2 * (qx * qx + qz * qz), m12 = 2 * (qy * qz - qw * qx);
        const R m20 = 2 * (qx * qz - qw * qy), m21 = 2 * (qy * qz + qw * qx), m22 = 1 - 2 * (qx * qx + qy * qy);
        for (int k = lane; k < D; k += 32) {
            const float4 e4 = sn[k];
            RayEnt<R> E{};
            E.cell = -1;
            if (__float_as_int(e4.w) & RS_ENTITY) {
                const R e[3] = {(R)e4.x, (R)e4.y, (R)e4.z};
                project_agent<R, true>(T, o, ag, e, &E.cell, &E.rn);
                const R dx = e[0] - o[0], dy = e[1] - o[1], dz = e[2] - o[2];
                E.bx = m00 * dx + m10 * dy + m20 * dz;
                E.by = m01 * dx + m11 * dy + m21 * dz;
                E.bz = m02 * dx + m12 * dy + m22 * dz;
                E.rel2 = dx * dx + dy * dy + dz * dz;
                const R r = (R)A.ray_r[k < T.n_lw ? 0 : 1];
                E.r2 = r * r;
                if (r > R(0)) E.box = E.rel2 <= E.r2 ? (N_THETA << 8) | (N_PHI << 24)
                                                     : ray_box((float)E.bx, (float)E.by, (float)E.bz, (float)sqrt(E.rel2), (float)r);
            }
            ent[k] = E;
        }
        for (int c = lane; c < N_CELLS; c += 32) { cur[c] = 1.0f; win[c] = -1; }
        __syncwarp();
        // entities in slot order, so that a cell's winner is decided by P4's sequential rule; the cells of one entity are
        // distinct, so the lanes never share a cell within an entity
        for (int k = 1; k < D; ++k) {
            const RayEnt<R> E = ent[k];
            if (E.cell < 0) continue;
            const int ti0 = E.box & 255, nti = (E.box >> 8) & 255, pj0 = (E.box >> 16) & 255, npj = (E.box >> 24) & 255;
            const int ct = E.cell / N_PHI, cp = E.cell - ct * N_PHI;
            const bool in_box = ct >= ti0 && ct < ti0 + nti && ((cp - pj0 + N_PHI) % N_PHI) < npj;
            for (int i = lane; i < nti * npj; i += 32) {
                const int ti = ti0 + i / npj, pj = (pj0 + i % npj) % N_PHI, c = ti * N_PHI + pj;
                double v = (double)ray_value<R>(E, ti, pj, inv_range);
                if (c == E.cell) v = fmin(v, E.rn);
                ray_offer(cur, win, c, v, k);
            }
            if (!in_box && lane == 0) ray_offer(cur, win, E.cell, E.rn, k);
            __syncwarp();
        }
        // the whole sphere: 3 x 338 floats, 8-byte aligned at every env (4,056 B rows), 16-byte stores from the first
        // 16-byte boundary on
        float* sph = A.obs_lidar + (long long)env * 3 * N_CELLS;
        auto val = [&](int f) {
            const int ch = f >= 2 * N_CELLS ? 2 : (f >= N_CELLS ? 1 : 0), c = f - ch * N_CELLS, w = win[c];
            if (ch == 0) return cur[c];
            if (w < 0) return 1.0f;
            return ch == 1 ? (float)((w < T.n_lw ? 3.0 : 1.0) / 5.0) : 0.1f;      // EntityType value / 5, age 1/10
        };
        const int head = (reinterpret_cast<uintptr_t>(sph) & 15) ? 2 : 0;
        const int n4 = (3 * N_CELLS - head) / 4;
        if (head && lane == 0) *reinterpret_cast<float2*>(sph) = make_float2(val(0), val(1));
        float4* s4 = reinterpret_cast<float4*>(sph + head);
        for (int i = lane; i < n4; i += 32) {
            const int f = head + 4 * i;
            s4[i] = make_float4(val(f), val(f + 1), val(f + 2), val(f + 3));
        }
        if (head + 4 * n4 < 3 * N_CELLS && lane == 0) {
            const int f = head + 4 * n4;
            *reinterpret_cast<float2*>(sph + f) = make_float2(val(f), val(f + 1));
        }
        if (A.lidar_ids) {
            int32_t* idp = A.lidar_ids + (long long)env * N_CELLS;           // 1,352 B rows: 8-byte stores if the base allows
            if (reinterpret_cast<uintptr_t>(idp) & 7) {                      // dc_buffers.lidar_ids need only be 4-byte aligned
                for (int c = lane; c < N_CELLS; c += 32) idp[c] = win[c];
            } else {
                int2* id2 = reinterpret_cast<int2*>(idp);
                for (int i = lane; i < N_CELLS / 2; i += 32) id2[i] = make_int2(win[2 * i], win[2 * i + 1]);
            }
        }
        __syncwarp();
    }
}

template <typename R> constexpr size_t ray_smem_bytes(int D) {
    return (size_t)RAY_ENV_WARPS * (N_CELLS * 8 + (size_t)D * sizeof(RayEnt<R>));
}

}  // namespace dc

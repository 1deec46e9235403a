// dronechase_b200 -- C ABI (include/dronechase_b200.h) over the sm_100a kernels.
// Build: nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo -shared -Xcompiler -fPIC
#include <cmath>
#include <algorithm>
#include "../../include/dronechase_b200.h"

#include <atomic>
#include <condition_variable>
#include <cstdio>
#include <functional>
#include <mutex>
#include <thread>
#include <vector>
#include <cstring>
#include <cstdlib>
#include <new>
#include <string>

#include "lidar_kernel.cuh"
#include "stage03.cuh"
#include "level5_stack.cuh"
#include "driven.cuh"
#include "raycast_env.cuh"

namespace {

thread_local std::string g_err;
std::atomic<uint64_t> g_launches{0};

int fail(int code, const std::string& msg) { g_err = msg; return code; }
int cuda_fail(cudaError_t e, const char* what) {
    g_err = std::string(what) + ": " + cudaGetErrorString(e);
    return DC_ERR_CUDA;
}
#define DC_CUDA(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return cuda_fail(e__, #call); } while (0)

// Host-side fork/join pool for the dc_host_scatter_* helpers.  Workers sleep on a condition variable between calls
// (no spinning): several ranks of one box share the host cores, and busy-waiting OpenMP teams of 8 ranks starved each
// other (r1p 8-GPU run: 50 ms per scatter call).
class HostPool {
public:
    static HostPool& get() { static HostPool* p = new HostPool; return *p; }      // never destroyed: workers outlive main()
    void run(int n_threads, int n_items, const std::function<void(int, int)>& fn) {
        if (n_threads > 64) n_threads = 64;
        if (n_threads <= 1 || n_items < 2 * n_threads) { fn(0, n_items); return; }
        std::unique_lock<std::mutex> call(call_mu_);              // one job at a time
        {
            std::lock_guard<std::mutex> lk(mu_);
            while ((int)workers_.size() < n_threads - 1) workers_.emplace_back([this, id = (int)workers_.size()] { loop(id); });
            fn_ = &fn; n_items_ = n_items; parts_ = n_threads; pending_ = n_threads - 1; ++epoch_;
            // dynamic chunks: on a shared box one descheduled thread would otherwise hold a static 1/n share of the
            // envs and everybody waits for it (4 threads 1.8 ms vs 8 threads 0.54 ms on the same call, e2e_breakdown4.txt)
            chunk_ = std::max(64, n_items / (n_threads * 8));
            next_.store(0, std::memory_order_relaxed);
        }
        cv_.notify_all();
        part(0);
        std::unique_lock<std::mutex> lk(mu_);
        done_.wait(lk, [this] { return pending_ == 0; });
        fn_ = nullptr;
    }
private:
    void part(int) {
        const int n = n_items_;
        for (;;) {
            const int c = next_.fetch_add(chunk_, std::memory_order_relaxed);
            if (c >= n) break;
            (*fn_)(c, std::min(c + chunk_, n));
        }
    }
    void loop(int id) {
        unsigned long long seen = 0;
        for (;;) {
            {
                std::unique_lock<std::mutex> lk(mu_);
                cv_.wait(lk, [&] { return epoch_ != seen; });
                seen = epoch_;
                if (id + 1 >= parts_) continue;                   // this job uses fewer threads
            }
            part(id + 1);
            std::lock_guard<std::mutex> lk(mu_);
            if (--pending_ == 0) done_.notify_one();
        }
    }
    std::mutex mu_, call_mu_;
    std::condition_variable cv_, done_;
    std::vector<std::thread> workers_;
    const std::function<void(int, int)>* fn_ = nullptr;
    int n_items_ = 0, parts_ = 1, pending_ = 0, chunk_ = 64;
    std::atomic<int> next_{0};
    unsigned long long epoch_ = 0;
};

}  // namespace

struct dc_sim {
    dc_config cfg;
    int device = 0;
    int D = 0, epb = 0, env_blocks = 0, env_threads = 0, dyn_blocks = 0, parity = 0;
    uint32_t div_m = 0;
    int epw = 32;
    int fam = dc::FAM_STAGE03;       // the step kernels' family instantiation (stage03.cuh FAM_*), see kernel_family
    bool quad_builtin = false;       // dc_config.quad is the built-in cf2x model (dyn_kernel<..., BUILTIN>)
    int gs = 1;                      // lanes per env in env_kernel's game-logic pass (stage03.cuh EnvCtx GS)
    long long n_slots = 0;
    size_t smem = 0, state_bytes = 0, env_bytes = 0, lw_bytes = 0, rsz = 4;
    void* state = nullptr;
    void* imu[2] = {nullptr, nullptr};
    int32_t* flagw = nullptr;
    unsigned char* nav = nullptr;
    void* agent = nullptr;
    int32_t* env = nullptr;
    double* lw_init = nullptr;
    int32_t* items[2] = {nullptr, nullptr};
    int32_t* count = nullptr;
    int2* sphere_desc = nullptr;
    double* last_dist = nullptr;
    int32_t* env5 = nullptr;         // level5 only (threatsense): per-env words, the agent's LiDAR ring, stacked-cell list
    float* ring_pose = nullptr;
    int32_t* ring_meta = nullptr;
    double* ring_feat = nullptr;
    int2* stack_prev = nullptr;
    int2* stack_prev2 = nullptr;     // student stack (dc_buffers.student_lidar), when student_hits is not bound
    int2* mo_prev = nullptr;         // multi-observer stacks (dc_buffers.mo_lidar), when mo_hits is not bound
    int32_t* mo_prev_n = nullptr;
    int2* lw_desc = nullptr;         // stage03 driven (dc_config.lw_driver): what dc_buffers.lw_lidar shows + Evaluation_Task.lw_kills
    int32_t* lw_kills = nullptr;
    bool raycast = false;            // dc_config.lidar == DC_LIDAR_RAYCAST: env_kernel<FAM_RAYCAST> + raycast_sphere_kernel
    float4* ray_snap = nullptr;      // env_kernel<FAM_RAYCAST>'s export of P4's inputs [E*D] (raycast_env.cuh)
    float ray_r[2] = {0.f, 0.f};     // dc_set_ray_radii: bounding radius of a wingman / of a munition
    bool reset_once = false;         // dc_reset has run: the radii are fixed from then on
    bool driven = false, has_nn = false;
    int mo_blocks = 0;
    int stack_blocks = 0;
    void* scratch = nullptr;     // parity harness only (dc_copy_state), allocated on first use
    dc_buffers buf{};
    bool bound = false;
    dc::TaskParams task{};
    dc::QuadParams<float> qf{};
    dc::QuadParams<double> qd{};
    // sub-batches (dc_config.sub_batches): a parent owns no device state, only its children and their streams
    std::vector<dc_sim*> kids;
    std::vector<int> kid_start;          // first env of each child
    std::vector<cudaStream_t> kid_stream;    // child 0 runs on the caller's stream
    std::vector<cudaEvent_t> kid_done;
    cudaEvent_t fork_ev = nullptr;
};

namespace {

template <typename R> dc::SimPtrs<R> sim_ptrs(const dc_sim* s) {
    dc::SimPtrs<R> p{};
    p.state = reinterpret_cast<dc::V4<R>*>(s->state);
    p.imu[0] = reinterpret_cast<dc::V4<R>*>(s->imu[0]); p.imu[1] = reinterpret_cast<dc::V4<R>*>(s->imu[1]);
    p.flagw = s->flagw; p.nav = s->nav; p.agent = reinterpret_cast<R*>(s->agent);
    p.env = s->env; p.lw_init = s->lw_init;
    p.items[0] = s->items[0]; p.items[1] = s->items[1]; p.count = s->count;
    p.sphere_desc = s->buf.lidar_hits ? reinterpret_cast<int2*>(s->buf.lidar_hits) : s->sphere_desc; p.last_dist = s->last_dist;
    p.env5 = s->env5; p.ring_pose = s->ring_pose; p.ring_meta = s->ring_meta; p.ring_feat = s->ring_feat;
    p.stack_prev = (s->cfg.family == DC_FAMILY_LEVEL5 && s->buf.lidar_hits) ? reinterpret_cast<int2*>(s->buf.lidar_hits) : s->stack_prev;
    p.mo_prev_n = s->mo_prev_n;
    p.lw_desc = s->lw_desc; p.lw_kills = s->lw_kills;
    return p;
}

template <typename R> dc::StepArgs<R> make_args(const dc_sim* s, const uint8_t* mask) {
    dc::StepArgs<R> a{};
    a.t = s->task;
    if constexpr (sizeof(R) == 4) a.q = s->qf; else a.q = s->qd;
    a.p = sim_ptrs<R>(s);
    a.parity = s->parity;
    a.actions = s->buf.actions; a.obs_lidar = s->buf.obs_lidar; a.obs_inertial = s->buf.obs_inertial;
    a.obs_last_action = s->buf.obs_last_action; a.reward = s->buf.reward; a.done = s->buf.done;
    a.info = s->buf.info; a.lidar_ids = s->buf.lidar_ids; a.term_inertial = s->buf.term_inertial;
    a.term_last_action = s->buf.term_last_action; a.stats = s->buf.stats; a.obs_mask = s->buf.obs_mask;
    a.mo_inertial = s->buf.mo_inertial; a.mo_last_action = s->buf.mo_last_action; a.mo_present = s->buf.mo_present;
    a.lw_actions = s->buf.lw_actions; a.lw_lidar = s->buf.lw_lidar; a.lw_inertial = s->buf.lw_inertial;
    a.lw_present = s->buf.lw_present; a.lw_info = s->buf.lw_info;
    a.reset_mask = mask; a.epb = s->epb; a.epw = s->epw; a.div_m = s->div_m;
    for (int i = 0; i < 10; ++i) {
        a.rk[2 * i] = s->task.k0 + (uint32_t)i * 0x9E3779B9u;
        a.rk[2 * i + 1] = s->task.k1 + (uint32_t)i * 0xBB67AE85u;
    }
    return a;
}

// level5: the stacked observation and, when dc_buffers.student_lidar is bound (base env), the second stack of the step
// that Level5Environment.compute_info puts into info["student_observation"] (level5_envrionment.py:291-292,342-346)
template <typename R> void launch_stacks(dc_sim* s, const dc::StepArgs<R>& a, cudaStream_t st) {
    if (s->cfg.level5_multi_obs == 2) return;      // Level52BTEvaluationEnvironment: no LiDAR is ever read
    if (s->cfg.level5_multi_obs) {
        // Level5DumbMultiObs: compute_observation returns zeros(1); the stacks are those of compute_info, one per wingman
        dc::StepArgs<R> b = a;
        b.obs_lidar = s->buf.mo_lidar; b.obs_mask = s->buf.mo_mask;
        b.p.stack_prev = s->buf.mo_hits ? reinterpret_cast<int2*>(s->buf.mo_hits) : s->mo_prev;
        dc::stack_kernel<R, dc::STACK_MULTI><<<s->mo_blocks, dc::STACK_WARPS * 32, 0, st>>>(b);
        g_launches.fetch_add(1, std::memory_order_relaxed);
        return;
    }
    dc::stack_kernel<R, dc::STACK_MAIN><<<s->stack_blocks, dc::STACK_WARPS * 32, 0, st>>>(a);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    if (s->buf.student_lidar) {
        dc::StepArgs<R> b = a;
        b.obs_lidar = s->buf.student_lidar; b.obs_mask = s->buf.student_mask;
        b.p.stack_prev = s->buf.student_hits ? reinterpret_cast<int2*>(s->buf.student_hits) : s->stack_prev2;
        dc::stack_kernel<R, dc::STACK_STUDENT><<<s->stack_blocks, dc::STACK_WARPS * 32, 0, st>>>(b);
        g_launches.fetch_add(1, std::memory_order_relaxed);
    }
}

#ifdef DC_PROFILE_PHASES
std::atomic<int> g_tl_seq{0};
int g_tl_sim[256];
#endif

// Step kernels are launched with programmatic stream serialisation (PDL): the next kernel's blocks are placed while the
// previous one drains -- dyn_kernel signals after its substep loop, env_kernel before its LiDAR pass -- and every step
// kernel starts with griddepcontrol.wait, which returns once the previous grid has completed and its writes are visible.
// What is hidden is the 3-6 us of launch latency between dependent kernels of one stream (profiles/r2t_timeline.txt).
template <typename A> cudaError_t launch_step(void (*kern)(const A), int grid, int block, size_t smem, cudaStream_t st, bool pdl, const A& a) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3((unsigned)block); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, a);
}

// The dyn_kernel instantiation: motor noise on or off, and (float32 only) the built-in cf2x model folded into the code
template <typename R, int FAM> auto dyn_kernel_for(bool noise, bool builtin) -> void (*)(const dc::StepArgs<R>) {
    if constexpr (sizeof(R) == 4 && FAM != dc::FAM_STAGE01) {
        if (builtin) return noise ? dc::dyn_kernel<R, true, FAM, true> : dc::dyn_kernel<R, false, FAM, true>;
    }
    return noise ? dc::dyn_kernel<R, true, FAM> : dc::dyn_kernel<R, false, FAM>;
}

// The env_kernel instantiation: gs = 8 lanes per env (swarm envs, stage03 only, see create_sim) or one
template <typename R, int MODE, int FAM> auto env_kernel_for(int gs) -> void (*)(const dc::StepArgs<R>) {
    if constexpr (FAM == dc::FAM_STAGE03) {
        if (gs == 8) return dc::env_kernel<R, MODE, FAM, 8>;
    }
    return dc::env_kernel<R, MODE, FAM>;
}

// env_kernel of a step or reset; a ray-cast sim (stage03 only) runs its FAM_RAYCAST instantiation and then rebuilds the
// agent's spheres
template <typename R, int MODE, int FAM> cudaError_t launch_env(dc_sim* s, const dc::StepArgs<R>& a, cudaStream_t st, bool pdl) {
    if constexpr (FAM == dc::FAM_STAGE03) {
        if (s->raycast) {
            dc::StepArgs<R> ea = a;
            ea.ray_snap = s->ray_snap;
            cudaError_t e = launch_step(s->gs == 8 ? dc::env_kernel<R, MODE, dc::FAM_RAYCAST, 8> : dc::env_kernel<R, MODE, dc::FAM_RAYCAST, 1>,
                                        s->env_blocks, s->env_threads, s->smem, st, pdl, ea);
            if (e != cudaSuccess) return e;
            dc::RaySphereArgs<R> ra{};
            ra.t = a.t; ra.agent = a.p.agent; ra.snap = s->ray_snap; ra.obs_lidar = a.obs_lidar; ra.lidar_ids = a.lidar_ids;
            ra.ray_r[0] = s->ray_r[0]; ra.ray_r[1] = s->ray_r[1];
            const int blocks = (s->cfg.n_envs + dc::RAY_ENV_WARPS - 1) / dc::RAY_ENV_WARPS;
            g_launches.fetch_add(1, std::memory_order_relaxed);
            return launch_step(dc::raycast_sphere_kernel<R>, blocks, dc::RAY_ENV_WARPS * 32, dc::ray_smem_bytes<R>(s->D), st, pdl, ra);
        }
    }
    return launch_step(env_kernel_for<R, MODE, FAM>(s->gs), s->env_blocks, s->env_threads, s->smem, st, pdl, a);
}

template <typename R, int FAM> int launch_family(dc_sim* s, int mode, const uint8_t* mask, cudaStream_t st) {
    dc::StepArgs<R> a = make_args<R>(s, mask);
    if (mode == dc::MODE_RESET) {
        // env_kernel<RESET> rebuilds the whole work list the next dyn_kernel reads
        DC_CUDA(cudaMemsetAsync(s->count + s->parity, 0, sizeof(int32_t), st));
        DC_CUDA((launch_env<R, dc::MODE_RESET, FAM>(s, a, st, false)));
        g_launches.fetch_add(1, std::memory_order_relaxed);
        if constexpr (dc::fam_l5(FAM)) launch_stacks<R>(s, a, st);
    } else {
#ifdef DC_PROFILE_PHASES
        a.tl_slot = g_tl_seq.fetch_add(2) & 255;      // dyn_kernel stamps row tl_slot, env_kernel row tl_slot + 1
        g_tl_sim[a.tl_slot] = g_tl_sim[a.tl_slot + 1] = (int)(((uintptr_t)s >> 4) & 0xffff);
#endif
#ifdef DC_PROFILE      // profiling builds only (nvcc -DDC_PROFILE): a product build cannot drop work from a timed step
        static const int skip = getenv("DC_SKIP") ? atoi(getenv("DC_SKIP")) : 0;
#else
        constexpr int skip = 0;
#endif
#ifdef DC_PROFILE
        static const int pdl = getenv("DC_PDL") ? atoi(getenv("DC_PDL")) : 2;
#else
        constexpr int pdl = 2;                 // 1: env_kernel only, 2: both step kernels
#endif
        if (skip != 1)
            DC_CUDA(launch_step(dyn_kernel_for<R, FAM>(s->cfg.quad[8] != 0.0, s->quad_builtin), s->dyn_blocks, dc::DYN_THREADS, 0,
                                st, pdl >= 2, a));
#ifdef DC_PROFILE_PHASES
        a.tl_slot += 1;
#endif
        if (skip != 2)
            DC_CUDA((launch_env<R, dc::MODE_STEP, FAM>(s, a, st, pdl >= 1)));
        g_launches.fetch_add(2, std::memory_order_relaxed);
        if constexpr (dc::fam_l5(FAM)) {
            if (skip == 0) launch_stacks<R>(s, a, st);
        }
        s->parity ^= 1;
    }
    DC_CUDA(cudaGetLastError());
    return DC_OK;
}

// The family instantiation of a config's step kernels: dc_config.family, except that the level5 multi-observer /
// evaluation envs and the stage03 tasks with policy-driven wingmen have kernels of their own
int kernel_family(const dc_config* cfg, bool driven) {
    if (cfg->family == DC_FAMILY_LEVEL5 && cfg->level5_multi_obs) return dc::FAM_L5_MULTI;
    if (cfg->family == DC_FAMILY_STAGE03 && driven) return dc::FAM_DRIVEN;
    return cfg->family;
}

template <typename R> int launch(dc_sim* s, int mode, const uint8_t* mask, cudaStream_t st) {
    switch (s->fam) {
        case dc::FAM_STAGE03: return launch_family<R, dc::FAM_STAGE03>(s, mode, mask, st);
        case dc::FAM_STAGE02: return launch_family<R, dc::FAM_STAGE02>(s, mode, mask, st);
        case dc::FAM_STAGE01: return launch_family<R, dc::FAM_STAGE01>(s, mode, mask, st);
        case dc::FAM_L5: return launch_family<R, dc::FAM_L5>(s, mode, mask, st);
        case dc::FAM_L5_MULTI: return launch_family<R, dc::FAM_L5_MULTI>(s, mode, mask, st);
        case dc::FAM_DRIVEN: return launch_family<R, dc::FAM_DRIVEN>(s, mode, mask, st);
    }
    return fail(DC_ERR_ARG, "launch: unknown kernel family");
}

template <typename R> int copy_drone_state(dc_sim* s, void* host, int to_device) {
    if (!s->scratch) DC_CUDA(cudaMalloc(&s->scratch, s->state_bytes));
    const int threads = 256;
    const int blocks = (int)((s->n_slots + threads - 1) / threads);
    dc::V4<R>* tmp = reinterpret_cast<dc::V4<R>*>(s->scratch);
    if (to_device) {
        DC_CUDA(cudaMemcpy(tmp, host, s->state_bytes, cudaMemcpyHostToDevice));
        dc::unpack_state_kernel<R><<<blocks, threads>>>(sim_ptrs<R>(s), s->parity, s->n_slots, tmp);
        DC_CUDA(cudaMemset(s->count + s->parity, 0, sizeof(int32_t)));
        dc::build_list_kernel<<<blocks, threads>>>(s->flagw, s->n_slots, s->items[s->parity], s->count + s->parity);
        g_launches.fetch_add(2, std::memory_order_relaxed);
        DC_CUDA(cudaDeviceSynchronize());
    } else {
        dc::pack_state_kernel<R><<<blocks, threads>>>(sim_ptrs<R>(s), s->parity, s->n_slots, tmp);
        g_launches.fetch_add(1, std::memory_order_relaxed);
        DC_CUDA(cudaDeviceSynchronize());
        DC_CUDA(cudaMemcpy(host, tmp, s->state_bytes, cudaMemcpyDeviceToHost));
    }
    return DC_OK;
}

}  // namespace

namespace {
// raycast_sphere_kernel's dynamic shared memory grows with the drones per env (ray_smem_bytes).  Its limit is an attribute of
// the function, shared by every sim of the process on the current device: it is raised past the 48 KB default only when a
// sim needs more, and never lowered, so creating a sim with fewer drones cannot make a larger sim's launches fail.
template <typename K> cudaError_t raise_ray_smem_limit(K* kern, size_t bytes) {
    if (bytes <= 48 * 1024) return cudaSuccess;
    static std::mutex mu;
    std::lock_guard<std::mutex> lk(mu);
    cudaFuncAttributes fa{};
    cudaError_t e = cudaFuncGetAttributes(&fa, kern);
    if (e != cudaSuccess || (size_t)fa.maxDynamicSharedSizeBytes >= bytes) return e;
    return cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
}

// Run f(child, stream) for every sub-batch: child 0 on the caller's stream, the others on their own streams,
// forked from and joined back into the caller's stream with events (also valid inside a stream capture).
template <typename F> int fork_join(dc_sim* s, cudaStream_t st, F f) {
    DC_CUDA(cudaEventRecord(s->fork_ev, st));
    int rc = DC_OK;
    for (size_t k = 1; k < s->kids.size() && rc == DC_OK; ++k) {
        DC_CUDA(cudaStreamWaitEvent(s->kid_stream[k], s->fork_ev, 0));
        rc = f(s->kids[k], s->kid_stream[k], (int)k);
        DC_CUDA(cudaEventRecord(s->kid_done[k], s->kid_stream[k]));
    }
    if (rc == DC_OK) rc = f(s->kids[0], st, 0);
    for (size_t k = 1; k < s->kids.size(); ++k) DC_CUDA(cudaStreamWaitEvent(st, s->kid_done[k], 0));
    return rc;
}
}  // namespace

extern "C" {

const char* dc_last_error(void) { return g_err.c_str(); }
uint64_t dc_launch_count(void) { return g_launches.load(); }

int dc_host_scatter_sphere(float* dense, const int32_t* prev_hits, const int32_t* hits, int32_t n_envs, int32_t n_drones,
                           int32_t n_lw, int32_t channels, int32_t n_threads) {
    if (!dense || !prev_hits || !hits) return fail(DC_ERR_ARG, "dc_host_scatter_sphere: null argument");
    if (n_envs < 1 || n_drones < 1 || (channels != 2 && channels != 3)) return fail(DC_ERR_ARG, "dc_host_scatter_sphere: bad sizes");
    if (n_threads < 1) n_threads = 1;
    const int per = channels * dc::N_CELLS;
    HostPool::get().run(n_threads, n_envs, [=](int e0, int e1) {
    constexpr int AHEAD = 6;                              // envs of look-ahead: the stores are random DRAM lines
    for (int e = e0; e < e1; ++e) {
        if (e + AHEAD < e1) {
            float* nsph = dense + (size_t)(e + AHEAD) * per;
            const int32_t* np_ = prev_hits + (size_t)(e + AHEAD) * n_drones * 2;
            const int32_t* nh = hits + (size_t)(e + AHEAD) * n_drones * 2;
            for (int d = 0; d < n_drones; ++d) {
                const int c0 = np_[2 * d], c1 = nh[2 * d];
                if (c0 == c1) { if (c1 >= 0 && c1 < dc::N_CELLS) __builtin_prefetch(nsph + c1, 1, 0); continue; }
                if (c0 >= 0 && c0 < dc::N_CELLS) for (int k = 0; k < channels; ++k) __builtin_prefetch(nsph + k * dc::N_CELLS + c0, 1, 0);
                if (c1 >= 0 && c1 < dc::N_CELLS) for (int k = 0; k < channels; ++k) __builtin_prefetch(nsph + k * dc::N_CELLS + c1, 1, 0);
            }
        }
        float* sph = dense + (size_t)e * per;
        const int32_t* p = prev_hits + (size_t)e * n_drones * 2;
        const int32_t* h = hits + (size_t)e * n_drones * 2;
        // A slot that still holds the cell it held in `prev` only needs its distance refreshed: the type and age
        // channels of that cell already carry this slot's values, and no other slot's un-write can name the cell
        // (a cell has one holder).  Entities cross a 0.24 rad cell border rarely, so this is the usual case.
        for (int d = 0; d < n_drones; ++d) {
            const int c = p[2 * d];
            if (c < 0 || c >= dc::N_CELLS || c == h[2 * d]) continue;
            sph[c] = 1.0f; sph[dc::N_CELLS + c] = 1.0f;
            if (channels == 3) sph[2 * dc::N_CELLS + c] = 1.0f;
        }
        for (int d = 0; d < n_drones; ++d) {
            const int c = h[2 * d];
            if (c < 0 || c >= dc::N_CELLS) continue;
            float rn; memcpy(&rn, h + 2 * d + 1, 4);
            sph[c] = rn;
            if (c == p[2 * d]) continue;
            sph[dc::N_CELLS + c] = d < n_lw ? 0.6f : 0.2f;
            if (channels == 3) sph[2 * dc::N_CELLS + c] = 0.1f;
        }
    }
    });
    return DC_OK;
}

int dc_host_scatter_stack(float* dense, const int32_t* prev_hits, const int32_t* hits, int32_t n_envs, int32_t n_drones,
                          int32_t n_threads) {
    if (!dense || !prev_hits || !hits) return fail(DC_ERR_ARG, "dc_host_scatter_stack: null argument");
    if (n_envs < 1 || n_drones < 1) return fail(DC_ERR_ARG, "dc_host_scatter_stack: bad sizes");
    if (n_threads < 1) n_threads = 1;
    const int cap = dc::STACK_MAX_SRC * n_drones + 1, per = DC_LIDAR_STACK * 3 * dc::N_CELLS;
    HostPool::get().run(n_threads, n_envs, [=](int e0, int e1) {
    constexpr int AHEAD = 4;
    for (int e = e0; e < e1; ++e) {
        if (e + AHEAD < e1) {
            float* nst = dense + (size_t)(e + AHEAD) * per;
            for (const int32_t* l : {prev_hits + (size_t)(e + AHEAD) * cap * 2, hits + (size_t)(e + AHEAD) * cap * 2})
                for (int i = 0; i < cap && l[2 * i] >= 0; ++i) {
                    const int code = l[2 * i] & 2047, sp = code / dc::N_CELLS, c = code - sp * dc::N_CELLS;
                    for (int k = 0; k < 3; ++k) __builtin_prefetch(nst + (sp * 3 + k) * dc::N_CELLS + c, 1, 0);
                }
        }
        float* st = dense + (size_t)e * per;
        const int32_t* p = prev_hits + (size_t)e * cap * 2;
        const int32_t* h = hits + (size_t)e * cap * 2;
        for (int i = 0; i < cap && p[2 * i] >= 0; ++i) {
            const int code = p[2 * i] & 2047, sp = code / dc::N_CELLS, c = code - sp * dc::N_CELLS;
            float* o = st + sp * 3 * dc::N_CELLS + c;
            o[0] = 1.0f; o[dc::N_CELLS] = 1.0f; o[2 * dc::N_CELLS] = 1.0f;
        }
        for (int i = 0; i < cap && h[2 * i] >= 0; ++i) {
            const int code = h[2 * i] & 2047, sp = code / dc::N_CELLS, c = code - sp * dc::N_CELLS;
            const int age = (h[2 * i] >> 12) & 15;
            float rn; memcpy(&rn, h + 2 * i + 1, 4);
            float* o = st + sp * 3 * dc::N_CELLS + c;
            o[0] = rn; o[dc::N_CELLS] = (h[2 * i] >> 11 & 1) ? 0.6f : 0.2f;
            o[2 * dc::N_CELLS] = age == 0 ? 0.1f : (float)((double)age / dc::RING);
        }
    }
    });
    return DC_OK;
}

static int create_sim(const dc_config* cfg, int device, dc_sim** out, bool allow_split);
int dc_create(const dc_config* cfg, int device, dc_sim** out) { return create_sim(cfg, device, out, true); }

static int create_sim(const dc_config* cfg, int device, dc_sim** out, bool allow_split) {
    if (!cfg || !out) return fail(DC_ERR_ARG, "dc_create: null argument");
    if (cfg->abi_version != DC_ABI_VERSION) return fail(DC_ERR_ARG, "dc_create: ABI version mismatch");
    if (cfg->n_envs < 1 || cfg->n_lw < 1 || cfg->n_lm < 1) return fail(DC_ERR_ARG, "dc_create: n_envs, n_lw, n_lm must be >= 1");
    if (cfg->n_lw + cfg->n_lm > 256) return fail(DC_ERR_ARG, "dc_create: at most 256 drones per env");
    if (cfg->initial_round < 1 || cfg->initial_round > cfg->n_lm) return fail(DC_ERR_ARG, "dc_create: initial_round outside [1, n_lm]");
    if (cfg->substeps < 1) return fail(DC_ERR_ARG, "dc_create: substeps must be >= 1");
    if (cfg->family < DC_FAMILY_STAGE03 || cfg->family > DC_FAMILY_LEVEL5) return fail(DC_ERR_ARG, "dc_create: unknown family");
    if (cfg->level5_multi_obs < 0 || cfg->level5_multi_obs > 2) return fail(DC_ERR_ARG, "dc_create: level5_multi_obs is 0, 1 or 2");
    if (cfg->level5_multi_obs && (cfg->family != DC_FAMILY_LEVEL5 || cfg->level5_base_env))
        return fail(DC_ERR_ARG, "dc_create: level5_multi_obs needs family level5 and excludes level5_base_env");
    if (cfg->family == DC_FAMILY_LEVEL5 && (cfg->n_lw > 8 || cfg->n_lw + cfg->n_lm > dc::STACK_MAX_D || cfg->initial_invaders < 1 || cfg->initial_invaders > cfg->n_lm ||
                                            cfg->invaders_per_round < 0 || cfg->max_rounds < 1 || cfg->lidar != DC_LIDAR_FUSED))
        return fail(DC_ERR_ARG, "dc_create: level5 needs n_lw <= 8, at most 64 drones, 1 <= initial_invaders <= n_lm, max_rounds >= 1, fused LiDAR");
    if (cfg->family == DC_FAMILY_STAGE01 && (cfg->n_lw != 2 || cfg->n_lm != 1))
        return fail(DC_ERR_ARG, "dc_create: stage01 is agent + idle wingman + one munition");
    bool driven = cfg->eval_task != 0, has_nn = false;
    for (int j = 0; j < 8; ++j) {
        const int d = cfg->lw_driver[j];
        if (d < DC_DRIVER_LEGACY || d > DC_DRIVER_NN_ALLY) return fail(DC_ERR_ARG, "dc_create: unknown lw_driver entry");
        if (d != DC_DRIVER_LEGACY && j >= cfg->n_lw) return fail(DC_ERR_ARG, "dc_create: lw_driver set for a wingman slot >= n_lw");
        driven |= d != DC_DRIVER_LEGACY;
        has_nn |= d == DC_DRIVER_NN || d == DC_DRIVER_NN_ALLY;
    }
    if (cfg->lidar == DC_LIDAR_RAYCAST && (cfg->family != DC_FAMILY_STAGE03 || driven))
        return fail(DC_ERR_ARG, "dc_create: the ray-cast LiDAR is built for the stage03 family without lw_driver / eval_task "
                                "(the agent's sphere only; level5 stacks, stage01/02 and policy-driven wingmen are not supported)");
    if (driven) {
        if (cfg->family != DC_FAMILY_STAGE03 || cfg->n_lw > 8 || cfg->lidar != DC_LIDAR_FUSED)
            return fail(DC_ERR_ARG, "dc_create: lw_driver / eval_task need family stage03, at most 8 wingmen and the fused LiDAR");
        if (cfg->n_lw + cfg->n_lm > dc::LWOBS_MAX_D) return fail(DC_ERR_ARG, "dc_create: too many drones for policy-driven wingmen");
        if (cfg->eval_task)
            for (int j = 0; j < cfg->n_lw; ++j)
                if (cfg->lw_driver[j] == DC_DRIVER_LEGACY || cfg->lw_driver[j] == DC_DRIVER_NN_ALLY)
                    return fail(DC_ERR_ARG, "dc_create: eval_task needs an NN, BT or STOP driver for every wingman");
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(DC_ERR_NO_DEVICE, "dc_create: no CUDA device visible (this library has no CPU fallback)");
    if (device < 0 || device >= ndev) return fail(DC_ERR_ARG, "dc_create: bad device index");
    DC_CUDA(cudaSetDevice(device));
    dc_sim* s = new (std::nothrow) dc_sim();
    if (!s) return fail(DC_ERR_ARG, "dc_create: out of host memory");
    s->cfg = *cfg; s->device = device;
    s->driven = driven; s->has_nn = has_nn;
    s->raycast = cfg->lidar == DC_LIDAR_RAYCAST;
    s->fam = kernel_family(cfg, driven);
    s->D = cfg->n_lw + cfg->n_lm;
    s->n_slots = (long long)cfg->n_envs * s->D;
    s->rsz = cfg->precision == DC_PRECISION_F64 ? 8 : 4;
    const bool level5 = cfg->family == DC_FAMILY_LEVEL5;
    // env_kernel geometry.  Each warp owns `epw` envs end to end; its slot passes walk epw * D slots 32 at a time, so
    // epw is sized for about 224 slots (7 trips, what D = 7 gives with 32 envs: measured best for D = 7, 11, 12 and 68,
    // gpurun_out/sweep_r1s_presets.txt).  A block is up to four such warps, its shared arrays (52 B per slot in
    // float32, 68 with the level5 features) under 48 KB.
    const int cap = (s->rsz == 8 ? 512 : 896) / (level5 ? 2 : 1) / s->D;
    int epw = (224 + s->D - 1) / s->D;
    if (epw > 32) epw = 32;
    if (epw > 1) epw &= ~1;                          // even: keeps the block's sphere slab 16 B aligned
    if (epw > cap) epw = cap > 1 ? (cap & ~1) : 1;
    if (epw < 1) epw = 1;
    int epb = epw * std::max(1, std::min(dc::ENV_THREADS / 32, cap / epw));
#ifdef DC_PROFILE
    if (const char* e = getenv("DC_EPW")) epw = std::max(1, std::min(std::min(32, cap), atoi(e)));
    if (const char* e = getenv("DC_EPB")) epb = std::max(1, std::min(cap, atoi(e)));
#endif
    if (epb > 1 && (epb & 1)) --epb;
    if (epb > cfg->n_envs) epb = cfg->n_envs;
    if (32 * ((epb + epw - 1) / epw) > dc::ENV_THREADS) epb = epw * (dc::ENV_THREADS / 32);
    s->epb = epb;
    s->env_blocks = (cfg->n_envs + epb - 1) / epb;
    s->epw = epw;
    // many drones per env (swarm): 8 lanes share an env's game logic, their O(drones) loops strided over the group
    s->gs = (s->fam == dc::FAM_STAGE03 && s->D >= 32 && epw <= 4) ? 8 : 1;
    s->env_threads = 32 * ((epb + epw - 1) / epw);
    s->div_m = (uint32_t)((1u << 20) / (unsigned)s->D + 1u);
    for (int i = 0; i < epb * s->D; ++i)
        if ((int)(((uint32_t)i * s->div_m) >> 20) != i / s->D || (uint64_t)i * s->div_m >> 32) {
            delete s;
            return fail(DC_ERR_ARG, "dc_create: envs per block x drones per env too large for the slot-index division");
        }
    s->dyn_blocks = (int)((s->n_slots + dc::DYN_THREADS - 1) / dc::DYN_THREADS);
    s->smem = dc::smem_bytes(epb * s->D, epb, s->rsz, level5);
    s->stack_blocks = (cfg->n_envs + dc::STACK_WARPS - 1) / dc::STACK_WARPS;
    s->state_bytes = (size_t)DC_STATE_QUADS * s->n_slots * 4 * s->rsz;
    s->env_bytes = (size_t)cfg->n_envs * DC_ENV_WORDS * 4;
    s->lw_bytes = (size_t)cfg->n_envs * cfg->n_lw * 3 * 8;
    {
        int K = allow_split ? cfg->sub_batches : 1;
#ifdef DC_PROFILE
        if (allow_split) if (const char* e = getenv("DC_SUB_BATCHES")) K = atoi(e);
#endif
        // two sub-batches: 0.115 -> 0.102 ms per 65,536-env step; four cost twice the host enqueue time for 0.103 (gpurun_out/sweep_r1r_i.txt)
        if (K <= 0) K = (s->rsz == 4 && cfg->n_envs >= 32768) ? 2 : 1;
        if (K > 16) K = 16;
        while (K > 1 && cfg->n_envs / K < 64) --K;
        if (K > 1) {
            // children of 64-env granularity (whole env_kernel warps, 16-byte aligned observation slabs)
            const int per = ((cfg->n_envs + K - 1) / K + 63) & ~63;
            cudaError_t ce = cudaEventCreateWithFlags(&s->fork_ev, cudaEventDisableTiming);
            for (int k = 0, start = 0; ce == cudaSuccess && start < cfg->n_envs; ++k, start += per) {
                dc_config c = *cfg;
                c.n_envs = std::min(per, cfg->n_envs - start);
                c.env_offset = cfg->env_offset + start;
                c.sub_batches = 1;
                dc_sim* kid = nullptr;
                const int rc = create_sim(&c, device, &kid, false);     // children never split again
                if (rc != DC_OK) { dc_destroy(s); return rc; }
                s->kids.push_back(kid); s->kid_start.push_back(start);
                cudaStream_t st = nullptr; cudaEvent_t ev = nullptr;
                if (k > 0) ce = cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking);
                if (ce == cudaSuccess) ce = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
                s->kid_stream.push_back(st); s->kid_done.push_back(ev);
            }
            if (ce != cudaSuccess) { dc_destroy(s); return cuda_fail(ce, "dc_create: sub-batch streams"); }
            *out = s;
            return DC_OK;
        }
    }
    dc::TaskParams& t = s->task;
    t.n_envs = cfg->n_envs; t.n_lw = cfg->n_lw; t.n_lm = cfg->n_lm; t.D = s->D;
    t.munition = cfg->munition; t.step_increment = cfg->step_increment; t.max_step = cfg->max_step;
    t.initial_round = cfg->initial_round; t.substeps = cfg->substeps; t.lm_nav = cfg->lm_nav;
    t.ally_mode = cfg->ally_mode; t.reward = cfg->reward;
    t.lidar = s->raycast ? DC_LIDAR_FUSED : cfg->lidar;      // env_kernel maintains the fused sphere the ray cast replaces
    t.fixed_lw_spawn = cfg->fixed_lw_spawn; t.auto_reset = cfg->auto_reset;
    t.family = cfg->family; t.support_munition = cfg->support_munition;
    t.initial_invaders = cfg->initial_invaders; t.invaders_per_round = cfg->invaders_per_round; t.max_rounds = cfg->max_rounds;
    t.n_rec = (level5 || s->driven) ? cfg->n_lw : 1;
    for (int j = 0; j < 8; ++j) t.lw_driver[j] = cfg->lw_driver[j];
    t.eval_task = cfg->eval_task != 0; t.time_limited = cfg->time_is_limited != 0;
    t.l5_base = level5 && cfg->level5_base_env != 0;
    t.l5_multi = level5 && cfg->level5_multi_obs != 0;
    t.l5_eval = level5 && cfg->level5_multi_obs == 2;
    t.respawn_r0 = cfg->respawn_r_min; t.respawn_r1 = cfg->respawn_r_max;
    t.env_offset = (uint32_t)cfg->env_offset;
    t.k0 = (uint32_t)(cfg->seed & 0xffffffffu); t.k1 = (uint32_t)(cfg->seed >> 32);
    t.dome = cfg->dome_radius; t.born = cfg->born_radius; t.lw_spawn = cfg->lw_spawn_radius;
    t.expl = cfg->explosion_range; t.shoot = cfg->shoot_range; t.cooldown = cfg->cooldown_steps;
    t.fire_p = cfg->fire_probability; t.lm_speed = cfg->lm_speed; t.bt_speed = cfg->bt_speed;
    t.ally_stop = cfg->ally_stop_mag; t.vel_bonus = cfg->vel_bonus;
    for (int k = 0; k < 3; ++k) t.building[k] = cfg->building[k];
    t.acos_born = t.born >= 4.0 ? std::acos(4.0 / t.born) : 0.0;
    t.acos_lw = t.lw_spawn >= 4.0 ? std::acos(4.0 / t.lw_spawn) : 0.0;
    s->qf = dc::make_quad<float>(cfg->quad); s->qd = dc::make_quad<double>(cfg->quad);
    s->quad_builtin = dc::quad_is_builtin(cfg->quad);
    const size_t imu_bytes = (size_t)s->n_slots * 4 * s->rsz, agent_bytes = (size_t)cfg->n_envs * t.n_rec * dc::AG_WORDS * s->rsz;
    cudaError_t e = cudaSuccess;
    auto alloc0 = [&](void** p, size_t bytes) {
        if (e == cudaSuccess) e = cudaMalloc(p, bytes);
        if (e == cudaSuccess) e = cudaMemset(*p, 0, bytes);
    };
    alloc0(&s->state, s->state_bytes);
    alloc0(&s->imu[0], imu_bytes); alloc0(&s->imu[1], imu_bytes);
    alloc0((void**)&s->flagw, (size_t)s->n_slots * 4); alloc0((void**)&s->nav, (size_t)s->n_slots);
    alloc0(&s->agent, agent_bytes);
    alloc0((void**)&s->env, s->env_bytes); alloc0((void**)&s->lw_init, s->lw_bytes);
    alloc0((void**)&s->items[0], (size_t)s->n_slots * 4); alloc0((void**)&s->items[1], (size_t)s->n_slots * 4);
    alloc0((void**)&s->count, 2 * sizeof(int32_t));
    alloc0((void**)&s->sphere_desc, (size_t)s->n_slots * sizeof(int2));
    alloc0((void**)&s->last_dist, (size_t)cfg->n_envs * cfg->n_lm * sizeof(double));
    if (level5) {
        const size_t entries = (size_t)cfg->n_envs * cfg->n_lw * dc::RING;
        alloc0((void**)&s->env5, (size_t)cfg->n_envs * dc::ENV5_WORDS * 4);
        alloc0((void**)&s->ring_pose, entries * 8 * sizeof(float));
        alloc0((void**)&s->ring_meta, entries * s->D * sizeof(int32_t));
        alloc0((void**)&s->ring_feat, entries * s->D * 3 * sizeof(double));
        alloc0((void**)&s->stack_prev, (size_t)cfg->n_envs * (dc::STACK_MAX_SRC * s->D + 1) * sizeof(int2));
        if (cfg->level5_base_env) {
            alloc0((void**)&s->stack_prev2, (size_t)cfg->n_envs * (dc::STACK_MAX_SRC * s->D + 1) * sizeof(int2));
            alloc0((void**)&s->mo_prev_n, (size_t)cfg->n_envs * sizeof(int32_t));
        }
        if (cfg->level5_multi_obs == 1) {
            const size_t n_obs = (size_t)cfg->n_envs * cfg->n_lw;
            alloc0((void**)&s->mo_prev, n_obs * (dc::STACK_MAX_SRC * s->D + 1) * sizeof(int2));
            alloc0((void**)&s->mo_prev_n, n_obs * sizeof(int32_t));
            s->mo_blocks = (int)((n_obs + dc::STACK_WARPS - 1) / dc::STACK_WARPS);
        }
    }
    if (s->driven) {
        const size_t n_obs = (size_t)cfg->n_envs * cfg->n_lw;
        alloc0((void**)&s->lw_kills, n_obs * sizeof(int32_t));
        if (e == cudaSuccess) e = cudaMalloc((void**)&s->lw_desc, n_obs * s->D * sizeof(int2));
        if (e == cudaSuccess) e = cudaMemset(s->lw_desc, 0xFE, n_obs * s->D * sizeof(int2));      // dc::LW_DESC_UNUSED
    }
    if (s->raycast) alloc0((void**)&s->ray_snap, (size_t)s->n_slots * sizeof(float4));
    if (e == cudaSuccess && s->raycast)
        e = s->rsz == 8 ? raise_ray_smem_limit(dc::raycast_sphere_kernel<double>, dc::ray_smem_bytes<double>(s->D))
                        : raise_ray_smem_limit(dc::raycast_sphere_kernel<float>, dc::ray_smem_bytes<float>(s->D));
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { dc_destroy(s); return cuda_fail(e, "dc_create: device allocation"); }
    *out = s;
    return DC_OK;
}

int dc_bind(dc_sim* s, const dc_buffers* b) {
    if (!s || !b) return fail(DC_ERR_ARG, "dc_bind: null argument");
    if (!b->actions || !b->obs_lidar || !b->obs_inertial || !b->obs_last_action || !b->reward || !b->done || !b->info)
        return fail(DC_ERR_ARG, "dc_bind: actions, obs_*, reward, done and info are mandatory");
    if ((reinterpret_cast<uintptr_t>(b->actions) | reinterpret_cast<uintptr_t>(b->obs_lidar) |
         reinterpret_cast<uintptr_t>(b->obs_last_action) | reinterpret_cast<uintptr_t>(b->info)) & 15)
        return fail(DC_ERR_ARG, "dc_bind: actions, obs_lidar, obs_last_action and info must be 16-byte aligned");
    if (s->cfg.family == DC_FAMILY_LEVEL5 && !b->obs_mask)
        return fail(DC_ERR_ARG, "dc_bind: level5 needs obs_mask ([E,6] validity mask of the stacked spheres in obs_lidar)");
    if (b->student_lidar || b->student_mask || b->student_hits) {
        if (!(s->cfg.family == DC_FAMILY_LEVEL5 && s->cfg.level5_base_env))
            return fail(DC_ERR_ARG, "dc_bind: student_* exist only with family level5 + level5_base_env (Level5Environment.compute_info)");
        if (!b->student_lidar || !b->student_mask)
            return fail(DC_ERR_ARG, "dc_bind: student_lidar and student_mask go together");
        if ((reinterpret_cast<uintptr_t>(b->student_lidar) & 15) || (reinterpret_cast<uintptr_t>(b->student_hits) & 7))
            return fail(DC_ERR_ARG, "dc_bind: student_lidar must be 16-byte, student_hits 8-byte aligned");
        if (s->bound && (s->buf.student_lidar != b->student_lidar || s->buf.student_hits != b->student_hits))
            return fail(DC_ERR_ARG, "dc_bind: student_lidar / student_hits carry state and cannot be re-bound to other buffers");
    } else if (s->bound && s->buf.student_lidar)
        return fail(DC_ERR_ARG, "dc_bind: student_lidar / student_hits carry state and cannot be re-bound to other buffers");
    if (s->cfg.family == DC_FAMILY_LEVEL5 && s->cfg.level5_multi_obs == 1) {
        if (!b->mo_lidar || !b->mo_mask || !b->mo_inertial || !b->mo_last_action || !b->mo_present)
            return fail(DC_ERR_ARG, "dc_bind: level5_multi_obs needs mo_lidar, mo_mask, mo_inertial, mo_last_action and mo_present");
        if ((reinterpret_cast<uintptr_t>(b->mo_lidar) | reinterpret_cast<uintptr_t>(b->mo_last_action)) & 15)
            return fail(DC_ERR_ARG, "dc_bind: mo_lidar and mo_last_action must be 16-byte aligned");
        if (reinterpret_cast<uintptr_t>(b->mo_hits) & 7) return fail(DC_ERR_ARG, "dc_bind: mo_hits must be 8-byte aligned");
        if (s->bound && (s->buf.mo_lidar != b->mo_lidar || s->buf.mo_hits != b->mo_hits || s->buf.mo_last_action != b->mo_last_action))
            return fail(DC_ERR_ARG, "dc_bind: mo_lidar / mo_hits / mo_last_action carry state and cannot be re-bound to other buffers");
    } else if (b->mo_lidar || b->mo_mask || b->mo_inertial || b->mo_last_action || b->mo_present || b->mo_hits)
        return fail(DC_ERR_ARG, "dc_bind: mo_* exist only with family level5 + level5_multi_obs == 1 (Level5DumbMultiObs.compute_info)");
    if (s->has_nn) {
        if (!b->lw_actions || !b->lw_lidar || !b->lw_inertial || !b->lw_present)
            return fail(DC_ERR_ARG, "dc_bind: policy-driven wingmen (dc_config.lw_driver) need lw_actions, lw_lidar, lw_inertial and lw_present");
        if ((reinterpret_cast<uintptr_t>(b->lw_actions) | reinterpret_cast<uintptr_t>(b->lw_info)) & 15)
            return fail(DC_ERR_ARG, "dc_bind: lw_actions and lw_info must be 16-byte aligned");
        if (s->bound && s->buf.lw_lidar != b->lw_lidar)
            return fail(DC_ERR_ARG, "dc_bind: lw_lidar carries state and cannot be re-bound to another buffer");
    } else if (b->lw_actions || b->lw_lidar || b->lw_inertial || b->lw_present)
        return fail(DC_ERR_ARG, "dc_bind: lw_actions / lw_lidar / lw_inertial / lw_present exist only with an NN driver in dc_config.lw_driver");
    if (b->lw_info && !s->driven) return fail(DC_ERR_ARG, "dc_bind: lw_info exists only with dc_config.lw_driver / eval_task");
    // obs_lidar is maintained incrementally (un-write of the remembered cells, then write): a different buffer would
    // never receive the hits it is supposed to show
    if (s->bound && (s->buf.obs_lidar != b->obs_lidar || s->buf.obs_mask != b->obs_mask))
        return fail(DC_ERR_ARG, "dc_bind: obs_lidar / obs_mask carry state and cannot be re-bound to other buffers");
    if (b->lidar_hits && s->bound && s->buf.lidar_hits != b->lidar_hits)
        return fail(DC_ERR_ARG, "dc_bind: lidar_hits carries state and cannot be re-bound to another buffer");
    if (b->lidar_hits && (reinterpret_cast<uintptr_t>(b->lidar_hits) & 7))
        return fail(DC_ERR_ARG, "dc_bind: lidar_hits must be 8-byte aligned");
    if (b->lidar_hits && s->cfg.lidar == DC_LIDAR_RAYCAST)
        return fail(DC_ERR_ARG, "dc_bind: lidar_hits cannot describe a ray-cast sphere (one (cell, r_n) per drone slot; a bounding "
                                "sphere covers several cells): leave it NULL with DC_LIDAR_RAYCAST");
    s->buf = *b; s->bound = true;
    for (size_t k = 0; k < s->kids.size(); ++k) {
        // a child sees its own rows of every [E, ...] tensor; stats is shared (atomics)
        const long long e0 = s->kid_start[k];
        const bool level5 = s->cfg.family == DC_FAMILY_LEVEL5;
        const long long lidar_row = (long long)(level5 ? DC_LIDAR_STACK * 3 : (s->cfg.lidar == DC_LIDAR_CLASSIC ? 2 : 3)) * dc::N_CELLS;
        const long long hits_row = (long long)(level5 ? dc::STACK_MAX_SRC * s->D + 1 : s->D) * 2;
        dc_buffers c = *b;
        c.actions = b->actions + e0 * 4;
        c.obs_lidar = b->obs_lidar + e0 * lidar_row;
        c.obs_inertial = b->obs_inertial + e0 * 15;
        c.obs_last_action = b->obs_last_action + e0 * 4;
        c.reward = b->reward + e0; c.done = b->done + e0; c.info = b->info + e0 * DC_INFO_WORDS;
        if (b->lidar_ids) c.lidar_ids = b->lidar_ids + e0 * dc::N_CELLS;
        if (b->term_inertial) c.term_inertial = b->term_inertial + e0 * 15;
        if (b->term_last_action) c.term_last_action = b->term_last_action + e0 * 4;
        if (b->obs_mask) c.obs_mask = b->obs_mask + e0 * DC_LIDAR_STACK;
        if (b->lidar_hits) c.lidar_hits = b->lidar_hits + e0 * hits_row;
        if (b->student_lidar) c.student_lidar = b->student_lidar + e0 * lidar_row;
        if (b->student_mask) c.student_mask = b->student_mask + e0 * DC_LIDAR_STACK;
        if (b->student_hits) c.student_hits = b->student_hits + e0 * hits_row;
        const long long L = s->cfg.n_lw;
        if (b->mo_lidar) c.mo_lidar = b->mo_lidar + e0 * L * lidar_row;
        if (b->mo_mask) c.mo_mask = b->mo_mask + e0 * L * DC_LIDAR_STACK;
        if (b->mo_inertial) c.mo_inertial = b->mo_inertial + e0 * L * 15;
        if (b->mo_last_action) c.mo_last_action = b->mo_last_action + e0 * L * 4;
        if (b->mo_present) c.mo_present = b->mo_present + e0 * L;
        if (b->mo_hits) c.mo_hits = b->mo_hits + e0 * L * hits_row;
        if (b->lw_actions) c.lw_actions = b->lw_actions + e0 * L * 4;
        if (b->lw_lidar) c.lw_lidar = b->lw_lidar + e0 * L * 3 * dc::N_CELLS;
        if (b->lw_inertial) c.lw_inertial = b->lw_inertial + e0 * L * 15;
        if (b->lw_present) c.lw_present = b->lw_present + e0 * L;
        if (b->lw_info) c.lw_info = b->lw_info + e0 * L * 4;
        const int rc = dc_bind(s->kids[k], &c);
        if (rc != DC_OK) return rc;
    }
    return DC_OK;
}



int dc_reset(dc_sim* s, const uint8_t* mask, void* stream) {
    if (!s) return fail(DC_ERR_ARG, "dc_reset: null sim");
    if (!s->bound) return fail(DC_ERR_UNBOUND, "dc_reset: call dc_bind first");
    s->reset_once = true;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    if (!s->kids.empty())
        return fork_join(s, st, [&](dc_sim* kid, cudaStream_t ks, int k) {
            return dc_reset(kid, mask ? mask + s->kid_start[k] : nullptr, ks); });
    return s->cfg.precision == DC_PRECISION_F64 ? launch<double>(s, dc::MODE_RESET, mask, st)
                                                : launch<float>(s, dc::MODE_RESET, mask, st);
}

int dc_step(dc_sim* s, void* stream) {
    if (!s) return fail(DC_ERR_ARG, "dc_step: null sim");
    if (!s->bound) return fail(DC_ERR_UNBOUND, "dc_step: call dc_bind first");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    if (!s->kids.empty())
        return fork_join(s, st, [&](dc_sim* kid, cudaStream_t ks, int) { return dc_step(kid, ks); });
    return s->cfg.precision == DC_PRECISION_F64 ? launch<double>(s, dc::MODE_STEP, nullptr, st)
                                                : launch<float>(s, dc::MODE_STEP, nullptr, st);
}

int dc_lw_observe(dc_sim* s, void* stream) {
    if (!s) return fail(DC_ERR_ARG, "dc_lw_observe: null sim");
    if (!s->bound) return fail(DC_ERR_UNBOUND, "dc_lw_observe: call dc_bind first");
    if (!s->has_nn) return fail(DC_ERR_ARG, "dc_lw_observe: no policy-driven wingman in dc_config.lw_driver");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    if (!s->kids.empty())
        return fork_join(s, st, [&](dc_sim* kid, cudaStream_t ks, int) { return dc_lw_observe(kid, ks); });
    const long long jobs = (long long)s->cfg.n_envs * s->cfg.n_lw;
    const int blocks = (int)((jobs + dc::LWOBS_WARPS - 1) / dc::LWOBS_WARPS);
    if (s->cfg.precision == DC_PRECISION_F64) dc::lw_obs_kernel<double><<<blocks, dc::LWOBS_WARPS * 32, 0, st>>>(make_args<double>(s, nullptr));
    else dc::lw_obs_kernel<float><<<blocks, dc::LWOBS_WARPS * 32, 0, st>>>(make_args<float>(s, nullptr));
    g_launches.fetch_add(1, std::memory_order_relaxed);
    DC_CUDA(cudaGetLastError());
    return DC_OK;
}

int dc_set_ray_radii(dc_sim* s, float r_lw, float r_lm) {
    if (!s) return fail(DC_ERR_ARG, "dc_set_ray_radii: null sim");
    if (s->cfg.lidar != DC_LIDAR_RAYCAST) return fail(DC_ERR_ARG, "dc_set_ray_radii: the sim was not created with DC_LIDAR_RAYCAST");
    if (!(r_lw >= 0.0f && r_lm >= 0.0f && std::isfinite(r_lw) && std::isfinite(r_lm)))
        return fail(DC_ERR_ARG, "dc_set_ray_radii: the radii must be finite and >= 0 (metres)");
    if (s->reset_once) return fail(DC_ERR_ARG, "dc_set_ray_radii: the radii are fixed once dc_reset has run");
    s->ray_r[0] = r_lw; s->ray_r[1] = r_lm;
    for (dc_sim* kid : s->kids) { kid->ray_r[0] = r_lw; kid->ray_r[1] = r_lm; }
    return DC_OK;
}

int dc_note_graph_replay(dc_sim* s) {
    if (!s) return fail(DC_ERR_ARG, "dc_note_graph_replay: null sim");
    for (dc_sim* kid : s->kids) kid->parity ^= 1;
    s->parity ^= 1;
    return DC_OK;
}

int dc_set_actions(dc_sim* s, const float* actions) {
    if (!s || !actions) return fail(DC_ERR_ARG, "dc_set_actions: null argument");
    if (reinterpret_cast<uintptr_t>(actions) & 15) return fail(DC_ERR_ARG, "dc_set_actions: actions must be 16-byte aligned");
    s->buf.actions = actions;
    for (size_t k = 0; k < s->kids.size(); ++k) s->kids[k]->buf.actions = actions + (long long)s->kid_start[k] * 4;
    return DC_OK;
}

void dc_destroy(dc_sim* s) {
    if (!s) return;
    for (dc_sim* kid : s->kids) dc_destroy(kid);
    for (cudaStream_t st : s->kid_stream) if (st) cudaStreamDestroy(st);
    for (cudaEvent_t ev : s->kid_done) if (ev) cudaEventDestroy(ev);
    if (s->fork_ev) cudaEventDestroy(s->fork_ev);
    cudaFree(s->state); cudaFree(s->imu[0]); cudaFree(s->imu[1]); cudaFree(s->flagw); cudaFree(s->nav);
    cudaFree(s->agent); cudaFree(s->env); cudaFree(s->lw_init); cudaFree(s->items[0]); cudaFree(s->items[1]);
    cudaFree(s->count); cudaFree(s->sphere_desc); cudaFree(s->last_dist); cudaFree(s->scratch);
    cudaFree(s->env5); cudaFree(s->ring_pose); cudaFree(s->ring_meta); cudaFree(s->ring_feat); cudaFree(s->stack_prev); cudaFree(s->stack_prev2); cudaFree(s->mo_prev); cudaFree(s->mo_prev_n); cudaFree(s->lw_desc); cudaFree(s->lw_kills);
    cudaFree(s->ray_snap);
    delete s;
}

size_t dc_state_bytes(const dc_sim* s, int which) {
    if (!s) return 0;
    return which == 0 ? s->state_bytes : which == 1 ? s->env_bytes : which == 2 ? s->lw_bytes : 0;
}

int dc_copy_state(dc_sim* s, int which, void* host, size_t bytes, int to_device) {
    if (!s || !host) return fail(DC_ERR_ARG, "dc_copy_state: null argument");
    if ((which != 0 && which != 1 && which != 2) || bytes != dc_state_bytes(s, which))
        return fail(DC_ERR_ARG, "dc_copy_state: bad selector or size");
    DC_CUDA(cudaSetDevice(s->device));
    DC_CUDA(cudaDeviceSynchronize());
    if (!s->kids.empty()) {
        // gather / scatter the children's blocks: which 0 is [quad][E*D][4], which 1 and 2 are env-major
        char* h = static_cast<char*>(host);
        for (size_t k = 0; k < s->kids.size(); ++k) {
            dc_sim* kid = s->kids[k];
            const size_t kb = dc_state_bytes(kid, which);
            const size_t e0 = (size_t)s->kid_start[k];
            if (which != 0) {
                const size_t row = bytes / (size_t)s->cfg.n_envs;
                const int rc = dc_copy_state(kid, which, h + e0 * row, kb, to_device);
                if (rc != DC_OK) return rc;
                continue;
            }
            std::vector<char> tmp(kb);
            const size_t qrow = 4 * s->rsz, big = (size_t)s->n_slots * qrow, small = (size_t)kid->n_slots * qrow, off = e0 * s->D * qrow;
            if (to_device) for (int q = 0; q < DC_STATE_QUADS; ++q) memcpy(tmp.data() + q * small, h + q * big + off, small);
            const int rc = dc_copy_state(kid, 0, tmp.data(), kb, to_device);
            if (rc != DC_OK) return rc;
            if (!to_device) for (int q = 0; q < DC_STATE_QUADS; ++q) memcpy(h + q * big + off, tmp.data() + q * small, small);
        }
        return DC_OK;
    }
    if (which == 0)
        return s->rsz == 8 ? copy_drone_state<double>(s, host, to_device) : copy_drone_state<float>(s, host, to_device);
    void* dev = which == 1 ? (void*)s->env : (void*)s->lw_init;
    DC_CUDA(cudaMemcpy(to_device ? dev : host, to_device ? host : dev, bytes,
                       to_device ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToHost));
    return DC_OK;
}

int dc_lidar_project(const float* pos, const float* quat, const int32_t* type, const uint8_t* alive,
                     const int32_t* obs_slot, int32_t n_envs, int32_t n_ent, int32_t n_obs,
                     int32_t flavour, double radius, float* sphere, int32_t* ids, void* stream) {
    if (!pos || !quat || !type || !alive || !obs_slot || !sphere) return fail(DC_ERR_ARG, "dc_lidar_project: null argument");
    if (n_envs < 1 || n_ent < 1 || n_ent > dc::LIDAR_MAX_ENT || n_obs < 1 || n_obs > n_ent)
        return fail(DC_ERR_ARG, "dc_lidar_project: need 1 <= n_obs <= n_ent <= 128");
    if (flavour != DC_LIDAR_FUSED && flavour != DC_LIDAR_CLASSIC) return fail(DC_ERR_ARG, "dc_lidar_project: bad flavour");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    dc::lidar_kernel<<<n_envs, dc::LIDAR_THREADS, 0, st>>>(pos, quat, type, alive, obs_slot, n_ent, n_obs, flavour,
                                                            radius, sphere, ids);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    DC_CUDA(cudaGetLastError());
    return DC_OK;
}

int dc_lidar_raycast(const float* pos, const float* quat, const float* radius_per_entity, const int32_t* type,
                     const uint8_t* alive, const int32_t* obs_slot, int32_t n_envs, int32_t n_ent, int32_t n_obs,
                     double max_range, float* sphere, int32_t* ids, void* stream) {
    if (!pos || !quat || !radius_per_entity || !type || !alive || !obs_slot || !sphere)
        return fail(DC_ERR_ARG, "dc_lidar_raycast: null argument");
    if (n_envs < 1 || n_ent < 1 || n_ent > dc::LIDAR_MAX_ENT || n_obs < 1 || n_obs > n_ent)
        return fail(DC_ERR_ARG, "dc_lidar_raycast: need 1 <= n_obs <= n_ent <= 128");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    dc::raycast_kernel<<<n_envs, dc::RAY_THREADS, 0, st>>>(pos, quat, radius_per_entity, type, alive, obs_slot, n_ent, n_obs,
                                                           max_range, sphere, ids);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    DC_CUDA(cudaGetLastError());
    return DC_OK;
}

int dc_scatter_hits(const int32_t* hits, const int64_t* row_index, int64_t n_rows, int32_t n_drones, int32_t n_lw,
                    int32_t channels, float* dense, void* stream) {
    if (!hits || !dense) return fail(DC_ERR_ARG, "dc_scatter_hits: null argument");
    if (n_rows < 0 || n_rows > 0x7fffffffLL || n_drones < 1 || (channels != 2 && channels != 3))
        return fail(DC_ERR_ARG, "dc_scatter_hits: bad sizes");
    if ((reinterpret_cast<uintptr_t>(hits) | reinterpret_cast<uintptr_t>(dense)) & 7)
        return fail(DC_ERR_ARG, "dc_scatter_hits: hits and dense must be 8-byte aligned");
    if (n_rows == 0) return DC_OK;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    dc::scatter_hits_kernel<<<(unsigned)n_rows, dc::SCATTER_THREADS, 0, st>>>(reinterpret_cast<const int2*>(hits),
                                                                             reinterpret_cast<const long long*>(row_index),
                                                                             n_drones, n_lw, channels, dense);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    DC_CUDA(cudaGetLastError());
    return DC_OK;
}

int dc_scatter_stack(const int32_t* hits, const int64_t* row_index, int64_t n_rows, int32_t n_drones, float* dense,
                     void* stream) {
    if (!hits || !dense) return fail(DC_ERR_ARG, "dc_scatter_stack: null argument");
    if (n_rows < 0 || n_rows > 0x7fffffffLL || n_drones < 1 || n_drones > dc::STACK_MAX_D)
        return fail(DC_ERR_ARG, "dc_scatter_stack: bad sizes");
    if ((reinterpret_cast<uintptr_t>(hits) & 7) || (reinterpret_cast<uintptr_t>(dense) & 15))
        return fail(DC_ERR_ARG, "dc_scatter_stack: hits must be 8-byte, dense 16-byte aligned");
    if (n_rows == 0) return DC_OK;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    dc::scatter_stack_kernel<<<(unsigned)n_rows, dc::SCATTER_THREADS, 0, st>>>(reinterpret_cast<const int2*>(hits),
                                                                              reinterpret_cast<const long long*>(row_index),
                                                                              dc::STACK_MAX_SRC * n_drones + 1, dense);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    DC_CUDA(cudaGetLastError());
    return DC_OK;
}

int dc_host_register(void* host, size_t bytes, void** device_ptr) {
    if (!host || !bytes || !device_ptr) return fail(DC_ERR_ARG, "dc_host_register: null argument");
    DC_CUDA(cudaHostRegister(host, bytes, cudaHostRegisterMapped | cudaHostRegisterPortable));
    const cudaError_t e = cudaHostGetDevicePointer(device_ptr, host, 0);
    if (e != cudaSuccess) { cudaHostUnregister(host); return cuda_fail(e, "cudaHostGetDevicePointer"); }
    return DC_OK;
}

int dc_host_unregister(void* host) {
    if (!host) return fail(DC_ERR_ARG, "dc_host_unregister: null argument");
    DC_CUDA(cudaHostUnregister(host));
    return DC_OK;
}

int dc_mirror_hits(int32_t* shown_hits, const int32_t* hits, int32_t n_envs, int32_t n_drones, int32_t n_lw, int32_t channels,
                   float* dense, void* stream) {
    if (!shown_hits || !hits || !dense) return fail(DC_ERR_ARG, "dc_mirror_hits: null argument");
    if (n_envs < 1 || n_drones < 1 || (channels != 2 && channels != 3)) return fail(DC_ERR_ARG, "dc_mirror_hits: bad sizes");
    if ((reinterpret_cast<uintptr_t>(shown_hits) | reinterpret_cast<uintptr_t>(hits)) & 7)
        return fail(DC_ERR_ARG, "dc_mirror_hits: hit lists must be 8-byte aligned");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    dc::mirror_hits_kernel<<<(n_envs + dc::MIRROR_THREADS - 1) / dc::MIRROR_THREADS, dc::MIRROR_THREADS, 0, st>>>(
        reinterpret_cast<int2*>(shown_hits), reinterpret_cast<const int2*>(hits), n_envs, n_drones, n_lw, channels, dense);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    DC_CUDA(cudaGetLastError());
    return DC_OK;
}

// hooks for the other translation units of the library (policy_kernel.cu): one error string, one launch counter
void dc_internal_set_error(const char* msg) { g_err = msg ? msg : ""; }
void dc_internal_count_launches(int n) { g_launches.fetch_add((uint64_t)n, std::memory_order_relaxed); }

size_t dc_abi_info(int which) {
    switch (which) {
        case 0: return DC_ABI_VERSION;
        case 1: return sizeof(dc_config);
        case 2: return sizeof(dc_buffers);
        default: return 0;
    }
}

int dc_diff_hits(int32_t* shown_hits, const int32_t* hits, int32_t n_envs, int32_t n_drones, int32_t n_lw, int32_t channels,
                 int32_t* out_pairs, void* stream) {
    if (!shown_hits || !hits || !out_pairs) return fail(DC_ERR_ARG, "dc_diff_hits: null argument");
    if (n_envs < 1 || n_drones < 1 || (channels != 2 && channels != 3)) return fail(DC_ERR_ARG, "dc_diff_hits: bad sizes");
    if ((long long)n_envs * channels * dc::N_CELLS > 0x7fffffffLL) return fail(DC_ERR_ARG, "dc_diff_hits: dense array too large for 32-bit indices");
    if ((reinterpret_cast<uintptr_t>(shown_hits) | reinterpret_cast<uintptr_t>(hits) | reinterpret_cast<uintptr_t>(out_pairs)) & 7)
        return fail(DC_ERR_ARG, "dc_diff_hits: buffers must be 8-byte aligned");
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    DC_CUDA(cudaMemsetAsync(out_pairs, 0, 8, st));
    dc::diff_hits_kernel<<<(n_envs + dc::MIRROR_THREADS - 1) / dc::MIRROR_THREADS, dc::MIRROR_THREADS, 0, st>>>(
        reinterpret_cast<int2*>(shown_hits), reinterpret_cast<const int2*>(hits), n_envs, n_drones, n_lw, channels,
        reinterpret_cast<int2*>(out_pairs));
    g_launches.fetch_add(1, std::memory_order_relaxed);
    DC_CUDA(cudaGetLastError());
    return DC_OK;
}

int dc_host_apply_pairs(float* dense, const int32_t* pairs, int64_t n_pairs, int32_t n_threads) {
    if (!dense || (!pairs && n_pairs > 0) || n_pairs < 0) return fail(DC_ERR_ARG, "dc_host_apply_pairs: bad argument");
    if (n_threads < 1) n_threads = 1;
    if (n_pairs > 0x7fffffffLL) return fail(DC_ERR_ARG, "dc_host_apply_pairs: too many pairs");
    int32_t* words = reinterpret_cast<int32_t*>(dense);
    auto body = [=](int i0, int i1) {
        constexpr int AHEAD = 24;                             // the stores are random DRAM lines: ask for them early
        for (int i = i0; i < i1; ++i) {
            if (i + AHEAD < i1) __builtin_prefetch(words + pairs[2 * (i + AHEAD)], 1, 0);
            words[pairs[2 * i]] = pairs[2 * i + 1];
        }
    };
    if (n_threads == 1 || n_pairs < 4096) body(0, (int)n_pairs);
    else HostPool::get().run(n_threads, (int)n_pairs, body);
    return DC_OK;
}

int dc_quad_is_builtin(const double* quad) { return quad && dc::quad_is_builtin(quad) ? 1 : 0; }

}  // extern "C"

#ifdef DC_PROFILE_PHASES
// rows of 4: sim tag, kernel (0 dyn, 1 env), first start, last end (globaltimer ns); reset = 1 clears the table first
extern "C" int dc_debug_timeline(long long* host, int reset) {
    unsigned long long t[256][2];
    if (reset) {
        for (int i = 0; i < 256; ++i) { t[i][0] = ~0ull; t[i][1] = 0; }
        g_tl_seq.store(0);
        return (int)cudaMemcpyToSymbol(dc::g_tl, t, sizeof(t));
    }
    const int rc = (int)cudaMemcpyFromSymbol(t, dc::g_tl, sizeof(t));
    for (int i = 0; i < 256; ++i) { host[4 * i] = g_tl_sim[i]; host[4 * i + 1] = i & 1; host[4 * i + 2] = (long long)t[i][0]; host[4 * i + 3] = (long long)t[i][1]; }
    return rc;
}
extern "C" int dc_debug_phase_clocks(long long* host, int n_warps) {
    return (int)cudaMemcpyFromSymbol(host, dc::g_phase_clk, sizeof(long long) * 8 * (size_t)n_warps);
}
#endif

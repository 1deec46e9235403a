// dronechase_b200 -- generalized advantage estimation over a device rollout (dc_gae).
//
// SB3's RolloutBuffer.compute_returns_and_advantage in DeviceRollout terms (dones[t] = the done AFTER step t, so SB3's
// episode_starts[t + 1] == dones[t]; the reference envs never truncate, so there is no bootstrap from a terminal observation):
//     delta_t = r_t + gamma * V_{t+1} * (1 - d_t) - V_t,  V_T = last_values
//     A_t = delta_t + gamma * lambda * (1 - d_t) * A_{t+1},  R_t = A_t + V_t
// One thread per env runs the reverse loop over T; the [T][E] reads and writes of a time step coalesce across the warp.
#include "../../include/dronechase_b200.h"

#include <cuda_runtime.h>
#include <cstdint>
#include <string>

extern "C" void dc_internal_set_error(const char* msg);
extern "C" void dc_internal_count_launches(int n);

namespace {

__global__ void __launch_bounds__(256) gae_kernel(const float* __restrict__ rewards, const uint8_t* __restrict__ dones,
                                                  const float* __restrict__ values, const float* __restrict__ last_values,
                                                  long long T, long long E, float gamma, float gl, float* __restrict__ adv,
                                                  float* __restrict__ ret) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= E) return;
    float next_v = last_values[e], a = 0.f;
    for (long long t = T - 1; t >= 0; --t) {
        const long long i = t * E + e;
        const float nonterminal = 1.f - (float)dones[i], v = values[i];
        const float delta = rewards[i] + gamma * next_v * nonterminal - v;
        a = delta + gl * nonterminal * a;
        adv[i] = a;
        ret[i] = a + v;
        next_v = v;
    }
}

int gfail(int code, const std::string& msg) { dc_internal_set_error(msg.c_str()); return code; }

}  // namespace

extern "C" int dc_gae(const float* rewards, const uint8_t* dones, const float* values, const float* last_values, int64_t T,
                      int64_t E, float gamma, float gae_lambda, float* advantages, float* returns, void* stream) {
    if (!rewards || !dones || !values || !last_values || !advantages || !returns || T < 0 || E < 0)
        return gfail(DC_ERR_ARG, "dc_gae: bad argument");
    if (!(gamma >= 0.f && gamma <= 1.f) || !(gae_lambda >= 0.f && gae_lambda <= 1.f))
        return gfail(DC_ERR_ARG, "dc_gae: gamma and gae_lambda must lie in [0, 1]");
    const long long blocks = (E + 255) / 256;
    if (blocks > 0x7fffffffLL) return gfail(DC_ERR_ARG, "dc_gae: too many envs for one launch");
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) { cudaGetLastError(); return gfail(DC_ERR_NO_DEVICE, "dc_gae: no CUDA device (there is no CPU fallback)"); }
    if (T == 0 || E == 0) return DC_OK;
    gae_kernel<<<(unsigned)blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(rewards, dones, values, last_values, T, E, gamma,
                                                                               gamma * gae_lambda, advantages, returns);
    dc_internal_count_launches(1);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return gfail(DC_ERR_CUDA, std::string("dc_gae: ") + cudaGetErrorString(e));
    return DC_OK;
}

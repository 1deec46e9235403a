// dronechase_b200 -- shared device helpers (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace dc {

constexpr int N_THETA = 13;
constexpr int N_PHI = 26;
constexpr int N_CELLS = N_THETA * N_PHI;
constexpr int STATE_QUADS = 13;
constexpr int ENV_WORDS = 16;
constexpr int INFO_WORDS = 8;

// ---- 4-wide state vectors: one 16 B (float) / 32 B (double) transaction per thread ----------
template <typename R> struct V4;
template <> struct __align__(16) V4<float> { float x, y, z, w; };
template <> struct __align__(32) V4<double> { double x, y, z, w; };

__device__ __forceinline__ V4<float> ld4(const V4<float>* p) {
    float4 t = *reinterpret_cast<const float4*>(p);
    return V4<float>{t.x, t.y, t.z, t.w};
}
__device__ __forceinline__ void st4(V4<float>* p, const V4<float>& v) {
    *reinterpret_cast<float4*>(p) = make_float4(v.x, v.y, v.z, v.w);
}
__device__ __forceinline__ V4<double> ld4(const V4<double>* p) {
    double2 a = reinterpret_cast<const double2*>(p)[0], b = reinterpret_cast<const double2*>(p)[1];
    return V4<double>{a.x, a.y, b.x, b.y};
}
__device__ __forceinline__ void st4(V4<double>* p, const V4<double>& v) {
    reinterpret_cast<double2*>(p)[0] = make_double2(v.x, v.y);
    reinterpret_cast<double2*>(p)[1] = make_double2(v.z, v.w);
}

// ---- scalar math, overloaded on the dynamics precision ------------------------------------
__device__ __forceinline__ float sqrt_(float x) { return sqrtf(x); }
__device__ __forceinline__ double sqrt_(double x) { return sqrt(x); }
// One MUFU each: the .ftz forms skip the denormal rescue (FSETP + 2 predicated FMUL per call) that rsqrtf / __fdividef
// carry without -ftz.  Every call site feeds them normal numbers (unit-quaternion norms, saturation ratios > 1, ...).
__device__ __forceinline__ float mufu_rsq(float x) { float r; asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float mufu_rcp(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float mufu_sqrt(float x) { float r; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float mufu_lg2(float x) { float r; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float rsqrt_(float x) { return mufu_rsq(x); }
__device__ __forceinline__ double rsqrt_(double x) { return 1.0 / sqrt(x); }
__device__ __forceinline__ float atan2_(float y, float x) { return atan2f(y, x); }
__device__ __forceinline__ double atan2_(double y, double x) { return atan2(y, x); }
__device__ __forceinline__ float asin_(float x) { return asinf(x); }
__device__ __forceinline__ double asin_(double x) { return asin(x); }
__device__ __forceinline__ void sincos_(float a, float* s, float* c) { sincosf(a, s, c); }
__device__ __forceinline__ void sincos_(double a, double* s, double* c) { sincos(a, s, c); }
__device__ __forceinline__ float log_(float x) { return logf(x); }
__device__ __forceinline__ double log_(double x) { return log(x); }
__device__ __forceinline__ float abs_(float x) { return fabsf(x); }
__device__ __forceinline__ double abs_(double x) { return fabs(x); }
__device__ __forceinline__ float min_(float a, float b) { return fminf(a, b); }
__device__ __forceinline__ double min_(double a, double b) { return fmin(a, b); }
__device__ __forceinline__ float max_(float a, float b) { return fmaxf(a, b); }
__device__ __forceinline__ double max_(double a, double b) { return fmax(a, b); }
__device__ __forceinline__ float fma_(float a, float b, float c) { return fmaf(a, b, c); }
__device__ __forceinline__ double fma_(double a, double b, double c) { return fma(a, b, c); }
__device__ __forceinline__ float fast_rcp(float x) { return mufu_rcp(x); }             // MUFU.RCP, 1 ulp
__device__ __forceinline__ double fast_rcp(double x) { return 1.0 / x; }
template <typename R> __device__ __forceinline__ R clamp_(R v, R lo, R hi) { return min_(max_(v, lo), hi); }

// ---- Philox4x32-10, same stream layout as oracle/philox.py ------------------------------------
// STREAM_POLICY: the Gaussian noise of the sampled actions (policy_kernel.cu, dc_policy_act; index = the caller's running counter)
enum { STREAM_HIT = 1, STREAM_SPAWN = 2, STREAM_MOTOR = 3, STREAM_FUSE = 4, STREAM_POLICY = 5 };

__device__ __forceinline__ uint4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                               uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
}

// The same block with the ten round keys precomputed by the host (StepArgs::rk: k0 + i * 0x9E3779B9, k1 + i * 0xBB67AE85
// interleaved): the key schedule was 20 uniform-datapath adds per call inside dyn_kernel's substep loop.
__device__ __forceinline__ uint4 philox4x32_10_rk(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, const uint32_t* rk) {
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        uint32_t n0 = hi1 ^ c1 ^ rk[2 * i], n2 = hi0 ^ c3 ^ rk[2 * i + 1];
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    }
    return make_uint4(c0, c1, c2, c3);
}

// one uniform on the 24-bit grid in [0,1): exact in fp32 and fp64
__device__ __forceinline__ double philox_uniform(uint32_t k0, uint32_t k1, uint32_t env, int stream,
                                                 uint32_t index, uint32_t sub = 0) {
    uint4 x = philox4x32_10(index, sub * 256u + (uint32_t)stream, env, 0u, k0, k1);
    return (double)(x.x >> 8) * (1.0 / 16777216.0);
}

}  // namespace dc

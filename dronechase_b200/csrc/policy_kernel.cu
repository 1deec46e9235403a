// dronechase_b200 -- the agent's policy network as ONE kernel (SURVEY.md section 8(f) rank 1, second half).
//
// The network is the reference's SB3 PPO actor with the LidarInertialActionExtractor
// (src/core/rl_framework/agents/policies/ppo_policies.py:234-342): Conv2d(C,32,k4,s4)-ReLU-Conv2d(32,64,k2,s2)-ReLU-Flatten over
// the (C,13,26) sphere, two 3 x 128 MLPs over the inertial vector and the last action, Linear(448, features_dim)-ReLU, the
// `pi` hidden layers (Tanh by default), action_net, clip to the action box = model.predict(obs, deterministic=True).
//
// One block = 64 envs, 16 warps (four warps per scheduler keep the tensor pipe fed; warp tiles of 32 rows x 32 columns for the
// wide layers, 16 x 32 for the 128-wide ones).  Every activation of
// those 64 envs lives in ONE shared-memory array act[64][452] from the sphere to the action: twelve layers, no HBM round trip between them (a layer-by-layer library path writes and re-reads
// 65,536 x 448 floats per layer).  Each layer is a [64 x K] x [K x N] product on the tensor cores (mma.sync m16n8k8 TF32,
// float32 accumulate); its outputs stay in the accumulator registers until every warp has finished reading the layer's
// input, so layers run in place.  Weights are re-laid out once (dc_policy_create) in the order the B fragments are consumed:
// one coalesced 8-byte load per lane, n-tile and k-step, served by L2 / L1 (the whole network is 1.7 MB).
// Row stride 452 words = 4 (mod 32): the four A-fragment words of a lane (rows g, g+8; columns t, t+4) and those of the
// other 31 lanes fall into 32 distinct banks.
// Precision: X3 = true splits both operands into a TF32 head and a TF32 tail and issues three MMAs (tail x head,
// head x tail, head x head): float32-grade products (the dropped tail x tail term is 2^-22 relative), which is what the
// parity tests compare with torch float32 at 2e-5; X3 = false is plain TF32 (10-bit mantissa operands, float32 accumulate),
// three times fewer MMAs, tested at 5e-3.
// Rows of the sphere that the second convolution never reads (conv1 output row 2: 13 // 4 = 3 rows, 3 // 2 = 1) are not computed.
//
// Actor-critic mode (policy_ac_kernel, dc_policy_act): the same trunk and pi branch, plus what SB3's collect_rollouts needs per
// step.  The features [64][F] are copied after final_layer into a stash stash[64][SV] behind red (SV = 260 = 4 mod 32, conflict-free
// A fragments like S; 66,560 B, 215,040 B of shared memory in all); the pi layers then run in place in act as in the plain kernel,
// and the vf layers of mlp_extractor.value_net run in place in the stash, the last one streamed into the 1-wide value_net head
// (partial sums in red, reused once the action head's have been added).  pi == (): final_layer is streamed into action_net, as
// in the plain kernel, and evaluated a second time into the stash.  The epilogue draws eps ~ N(0, I) (Box-Muller on one Philox
// block per env: STREAM_POLICY), raw = mean + exp(log_std) * eps, env_action = clip(raw), log_prob of raw under the diagonal
// Gaussian; with sample = 0 the action is the plain kernel's clipped mean, bit for bit.
#include "../../include/dronechase_b200.h"
#include "common.cuh"

#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <new>
#include <string>
#include <vector>

extern "C" void dc_internal_set_error(const char* msg);
extern "C" void dc_internal_count_launches(int n);

namespace dcp {

constexpr int BM = 64, WARPS = 16, THREADS = 32 * WARPS, S = 452, MAX_LAYERS = 16, MAX_CHUNKS = 16;
#ifndef DCP_WIDE
#define DCP_WIDE 1                 // 32-row x 32-column warp tiles for the wide layers (a B fragment serves two m-tiles: 20 % fewer
                                   // operand bytes through L1 per MMA than 16 x 64; 0 = 16 x 64 tiles.  profiles/r2av_variants.txt)
#endif
#ifndef DCP_PF_TF32
#define DCP_PF_TF32 2              // k-steps of B fragments in flight per warp, TF32 mode (3 and 4 measured the same: r2av)
#endif
#ifndef DCP_PF_X3
#define DCP_PF_X3 1                // the same, 3xTF32 mode (head + tail fragments)
#endif
constexpr int MAX_UNITS = 32;      // partial sums of the head: one per 32-column unit of the last layer (1024 / 32)
constexpr int SMEM_BYTES = (BM * S + MAX_UNITS * BM * 4) * 4;
constexpr int PAD_STEPS = 4;       // k-steps of 8 n-tiles behind the packed weights that the prefetch may touch
constexpr int SV = 260;            // row stride of the actor-critic kernel's feature stash (features_dim <= 256)
constexpr int SMEM_AC_BYTES = SMEM_BYTES + BM * SV * 4;
constexpr int FINAL_LAYER = 6;     // layers[6] = final_layer (after the three inertial and three last-action layers)
constexpr int MAX_VF = 8;
enum { ACT_NONE = 0, ACT_RELU = 1, ACT_TANH = 2 };
enum { SRC_SMEM = 0, SRC_INERTIAL = 1, SRC_ACTION = 2 };

struct Layer {
    int K, KS, N, in_off, out_off, act, src;
    int w_off;          // first float2 of the packed weights
    int b_off;          // first float of the bias in Params::fp
};

struct Params {
    const float2* w_hi;
    const float2* w_lo;
    const float* fp;                 // biases, head weights [4][N_last], head bias
    const float* lidar;
    const float* inertial;
    const float* last_action;
    float* actions;
    long long n_envs;
    int C, n_layers;                 // layers[0 .. n_layers-2]: dense; layers[n_layers-1]: the last hidden layer, fused with the head
    int conv1_w, conv1_b, conv2_w, conv2_b, head_w, head_b;
    float low[4], high[4];
    Layer layers[MAX_LAYERS];
};

// The actor-critic kernel's parameters: the plain kernel's (p.actions = the clipped env actions) + the value branch + sampling.
struct ACParams {
    Params p;
    Layer vf[MAX_VF];                // mlp_extractor.value_net: in and out in the stash; vf[n_vf-1] is streamed into value_net
    int n_vf, value_w, value_b, log_std;     // offsets in p.fp
    float* raw;                      // [n][4] unclipped samples (sample = 1)
    float* log_prob;                 // [n] (sample = 1)
    float* value;                    // [n]
    uint32_t k0, k1, env_offset, counter;
    int sample;
};

__device__ __forceinline__ uint32_t tf32_rna(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return r;
}

__device__ __forceinline__ void mma_tf32(float (&d)[4], const uint32_t (&a)[4], float b0, float b1) {
    asm("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(__float_as_uint(b0)), "r"(__float_as_uint(b1)));
}

// X3 = false: MUFU.TANH (2^-11 relative, inside the TF32 mode's 5e-3) and the value rounded to TF32 where it is produced, so
// that the MMA loops pass activation words to the tensor cores as they are (cvt.rna.tf32 is a four-instruction sequence on
// sm_100a; inputs read from global memory -- sphere, inertial vector, last action -- are truncated by the hardware instead).
template <bool X3>
__device__ __forceinline__ float activate(float x, int act) {
    float y = x;
    if (act == ACT_RELU) y = fmaxf(x, 0.f);
    else if (act == ACT_TANH) {
        if (X3) y = tanhf(x);
        else asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    }
    return X3 ? y : __uint_as_float(tf32_rna(y));
}

// X3: a = head + tail exactly, head = the TF32 the hardware would read anyway (low 13 bits cleared), tail = the rest
template <bool X3>
__device__ __forceinline__ void split_a(const float (&a)[4], uint32_t (&hi)[4], uint32_t (&lo)[4]) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        hi[i] = X3 ? (__float_as_uint(a[i]) & 0xffffe000u) : __float_as_uint(a[i]);
        lo[i] = X3 ? __float_as_uint(a[i] - __uint_as_float(hi[i])) : 0u;
    }
}

// acc[mt][j] += A(m-tile mt) x B(n-tile nt0 + j) over KS k-steps of 8.  aload(mt, ks, a) delivers the lane's four A words
// (rows g, g+8, g, g+8; columns t, t, t+4, t+4 of the k-step).  The B fragments come from L2 (L1 for all but the first of the
// four row-group warps of a column chunk): they are requested PF k-steps ahead -- a k-step of a warp is only 8 MMAs (~70 cycles
// of its scheduler's tensor pipe, measured 0.467 m16n8k8 MMAs per cycle and SM: profiles/r2ao_mma_rate.txt), so one step of
// lead does not cover an L2 round trip.  X3: three sweeps over the accumulators (tail x head, head x tail, head x head),
// so that MMAs into the same accumulator are MT*NT apart instead of back to back.
template <int MT, int NT, int NTG, bool X3, class ALoad>
__device__ __forceinline__ void mma_block(float (&acc)[MT][NT][4], ALoad&& aload, int KS, const float2* __restrict__ whi,
                                          const float2* __restrict__ wlo, int nt0, int lane) {
    constexpr int PF = X3 ? DCP_PF_X3 : DCP_PF_TF32;
    // packed weights: [group of NT n-tiles][k-step][n-tile in group][lane] -- one pointer per operand, immediate offsets
    // (a warp consumes NT n-tiles of a packed group of NTG)
    const float2* ph = whi + (size_t)(nt0 / NTG) * KS * (NTG * 32) + (nt0 % NTG) * 32 + lane;
    const float2* pl = wlo + (size_t)(nt0 / NTG) * KS * (NTG * 32) + (nt0 % NTG) * 32 + lane;
    float2 qh[PF][NT], ql[PF][NT];
    // (requests run up to PF k-steps past the end of the group: into the next group or the PAD_STEPS of padding behind the
    // last one -- never used, and no clamp in the address arithmetic)
#pragma unroll
    for (int s = 0; s < PF; ++s) {
#pragma unroll
        for (int j = 0; j < NT; ++j) {
            qh[s][j] = __ldg(ph + s * (NTG * 32) + j * 32);
            ql[s][j] = X3 ? __ldg(pl + s * (NTG * 32) + j * 32) : make_float2(0.f, 0.f);
        }
    }
    for (int ks0 = 0; ks0 < KS; ks0 += PF) {
#pragma unroll
        for (int s = 0; s < PF; ++s) {
            const int ks = ks0 + s;
            if (ks < KS) {
                uint32_t ah[MT][4], al[MT][4];
#pragma unroll
                for (int mt = 0; mt < MT; ++mt) {
                    float a[4];
                    aload(mt, ks, a);
                    split_a<X3>(a, ah[mt], al[mt]);
                }
                if (X3) {
#pragma unroll
                    for (int j = 0; j < NT; ++j)
#pragma unroll
                        for (int mt = 0; mt < MT; ++mt) mma_tf32(acc[mt][j], al[mt], qh[s][j].x, qh[s][j].y);
#pragma unroll
                    for (int j = 0; j < NT; ++j)
#pragma unroll
                        for (int mt = 0; mt < MT; ++mt) mma_tf32(acc[mt][j], ah[mt], ql[s][j].x, ql[s][j].y);
                }
#pragma unroll
                for (int j = 0; j < NT; ++j)
#pragma unroll
                    for (int mt = 0; mt < MT; ++mt) mma_tf32(acc[mt][j], ah[mt], qh[s][j].x, qh[s][j].y);
                // this stage's registers are free again: request k-step ks + PF into them (no copies)
#pragma unroll
                for (int j = 0; j < NT; ++j) {
                    qh[s][j] = __ldg(ph + (ks + PF) * (NTG * 32) + j * 32);
                    ql[s][j] = X3 ? __ldg(pl + (ks + PF) * (NTG * 32) + j * 32) : make_float2(0.f, 0.f);
                }
            }
        }
    }
}

// One dense layer over the block's 64 rows: a warp owns 16*MT rows x NT*8 columns, chosen per width so that the 16 warps all
// have a tile.  Outputs are written after a barrier, so in_off / out_off may overlap.  The input rows are `in` (row stride LDI),
// the outputs `out` (row stride LDO): act for the plain kernel, the stash for the value branch.
template <int MT, int NT, bool X3, int LDI = S, int LDO = S>
__device__ __forceinline__ void dense_layer(const float* in, float* out, const Layer& L, const Params& P, long long env0, int warp, int lane) {
    constexpr int RG = BM / (16 * MT);
    const int g = lane >> 2, t = lane & 3;
    const int rg = warp % RG, cc = warp / RG;
    const int row0 = rg * 16 * MT, nt0 = cc * NT;
    const bool active = nt0 * 8 < L.N;
    float acc[MT][NT][4];
#pragma unroll
    for (int mt = 0; mt < MT; ++mt)
#pragma unroll
        for (int j = 0; j < NT; ++j)
#pragma unroll
            for (int i = 0; i < 4; ++i) acc[mt][j][i] = 0.f;
    if (active) {
        const float2* wh = P.w_hi + L.w_off;
        const float2* wl = P.w_lo + L.w_off;
        if (L.src == SRC_SMEM) {
            const float* base = in + (row0 + g) * LDI + L.in_off + t;
            mma_block<MT, NT, 8, X3>(acc, [&](int mt, int ks, float (&a)[4]) {
                const float* p = base + mt * 16 * LDI + ks * 8;
                a[0] = p[0]; a[1] = p[8 * LDI]; a[2] = p[4]; a[3] = p[8 * LDI + 4];
            }, L.KS, wh, wl, nt0, lane);
        } else {
            const float* src = L.src == SRC_INERTIAL ? P.inertial : P.last_action;
            const int ld = L.K;
            mma_block<MT, NT, 8, X3>(acc, [&](int mt, int ks, float (&a)[4]) {
                const long long ea = env0 + row0 + mt * 16 + g, eb = ea + 8;
                const int k0 = ks * 8 + t, k1 = k0 + 4;
                a[0] = (ea < P.n_envs && k0 < ld) ? __ldg(src + ea * ld + k0) : 0.f;
                a[1] = (eb < P.n_envs && k0 < ld) ? __ldg(src + eb * ld + k0) : 0.f;
                a[2] = (ea < P.n_envs && k1 < ld) ? __ldg(src + ea * ld + k1) : 0.f;
                a[3] = (eb < P.n_envs && k1 < ld) ? __ldg(src + eb * ld + k1) : 0.f;
            }, L.KS, wh, wl, nt0, lane);
        }
    }
    __syncthreads();                                    // every warp has read the layer's input
    if (active) {
#pragma unroll
        for (int mt = 0; mt < MT; ++mt)
#pragma unroll
            for (int j = 0; j < NT; ++j) {
                const int col = (nt0 + j) * 8 + 2 * t;
                const float b0 = __ldg(P.fp + L.b_off + col), b1 = __ldg(P.fp + L.b_off + col + 1);
                float* o = out + (row0 + mt * 16 + g) * LDO + L.out_off + col;
                *reinterpret_cast<float2*>(o) = make_float2(activate<X3>(acc[mt][j][0] + b0, L.act), activate<X3>(acc[mt][j][1] + b1, L.act));
                *reinterpret_cast<float2*>(o + 8 * LDO) = make_float2(activate<X3>(acc[mt][j][2] + b0, L.act), activate<X3>(acc[mt][j][3] + b1, L.act));
            }
    }
    __syncthreads();
}

// The last hidden layer, never stored: activation(.) goes straight into the NH sums of the head (action_net: 4, value_net: 1),
// whose weights [NH][N] are at P.fp + hw_off.  Passes of 256 columns; a warp owns 16*MT rows x NT*8 columns (one `unit`); its
// partial sums go to red[unit][row][output] and are added in unit order at the end.  Input rows: `in`, row stride LD.
template <int MT, int NT, bool X3, int NH = 4, int LD = S>
__device__ __forceinline__ void head_layer(const float* in, float* red, const Layer& L, const Params& P, int hw_off, int warp, int lane) {
    constexpr int RG = BM / (16 * MT), CP = WARPS / RG;   // column units per pass
    const int g = lane >> 2, t = lane & 3;
    const int rg = warp % RG, cc = warp / RG;
    const int row0 = rg * 16 * MT;
    const float* base = in + (row0 + g) * LD + L.in_off + t;
    const float* hw = P.fp + hw_off;
    const int n_units = L.N / (NT * 8);
    for (int pass = 0; pass * CP < n_units; ++pass) {
        const int unit = pass * CP + cc;
        if (unit < n_units) {
            float acc[MT][NT][4];
#pragma unroll
            for (int mt = 0; mt < MT; ++mt)
#pragma unroll
                for (int j = 0; j < NT; ++j)
#pragma unroll
                    for (int i = 0; i < 4; ++i) acc[mt][j][i] = 0.f;
            mma_block<MT, NT, 8, X3>(acc, [&](int mt, int ks, float (&a)[4]) {
                const float* p = base + mt * 16 * LD + ks * 8;
                a[0] = p[0]; a[1] = p[8 * LD]; a[2] = p[4]; a[3] = p[8 * LD + 4];
            }, L.KS, P.w_hi + L.w_off, P.w_lo + L.w_off, unit * NT, lane);
            float part[MT][2][NH];                       // [m-tile][row g / g+8][output]
#pragma unroll
            for (int mt = 0; mt < MT; ++mt)
#pragma unroll
                for (int h = 0; h < 2; ++h)
#pragma unroll
                    for (int k = 0; k < NH; ++k) part[mt][h][k] = 0.f;
#pragma unroll
            for (int j = 0; j < NT; ++j) {
                const int col = (unit * NT + j) * 8 + 2 * t;
                const float b0 = __ldg(P.fp + L.b_off + col), b1 = __ldg(P.fp + L.b_off + col + 1);
                float w0[NH], w1[NH];
#pragma unroll
                for (int k = 0; k < NH; ++k) { w0[k] = __ldg(hw + k * L.N + col); w1[k] = __ldg(hw + k * L.N + col + 1); }
#pragma unroll
                for (int mt = 0; mt < MT; ++mt) {
                    const float h00 = activate<X3>(acc[mt][j][0] + b0, L.act), h01 = activate<X3>(acc[mt][j][1] + b1, L.act);
                    const float h10 = activate<X3>(acc[mt][j][2] + b0, L.act), h11 = activate<X3>(acc[mt][j][3] + b1, L.act);
#pragma unroll
                    for (int k = 0; k < NH; ++k) {
                        part[mt][0][k] = fmaf(h00, w0[k], fmaf(h01, w1[k], part[mt][0][k]));
                        part[mt][1][k] = fmaf(h10, w0[k], fmaf(h11, w1[k], part[mt][1][k]));
                    }
                }
            }
#pragma unroll
            for (int mt = 0; mt < MT; ++mt)
#pragma unroll
                for (int h = 0; h < 2; ++h)
#pragma unroll
                    for (int k = 0; k < NH; ++k) {
                        float v = part[mt][h][k];
                        v += __shfl_xor_sync(0xffffffffu, v, 1);
                        v += __shfl_xor_sync(0xffffffffu, v, 2);
                        if (t == 0) red[(unit * BM + row0 + mt * 16 + h * 8 + g) * NH + k] = v;
                    }
        }
    }
}

// The value of each of the block's rows for the actor-critic kernel, returned to the threads (row = tid / 4, any k) of the
// epilogue; features in the stash (pi != ()) or still to be computed from act (pi == ()); red is free.
template <bool X3>
__device__ __forceinline__ float value_branch(const float* act, float* stash, float* red, const Params& P, const ACParams& A,
                                              long long env0, int tid, int warp, int lane) {
    constexpr int UNIT = DCP_WIDE ? 32 : 64;
    if (P.n_layers == FINAL_LAYER + 1) {                 // pi == (): the plain kernel never stores the features
        const Layer& L = P.layers[FINAL_LAYER];
        if (L.N == 128 || L.N == 64) dense_layer<1, 4, X3, S, SV>(act, stash, L, P, env0, warp, lane);
        else if (DCP_WIDE) dense_layer<2, 4, X3, S, SV>(act, stash, L, P, env0, warp, lane);
        else dense_layer<1, 8, X3, S, SV>(act, stash, L, P, env0, warp, lane);
    }
    for (int li = 0; li + 1 < A.n_vf; ++li) {
        const Layer& L = A.vf[li];
        if (L.N == 128 || L.N == 64) dense_layer<1, 4, X3, SV, SV>(stash, stash, L, P, env0, warp, lane);
        else if (DCP_WIDE) dense_layer<2, 4, X3, SV, SV>(stash, stash, L, P, env0, warp, lane);
        else dense_layer<1, 8, X3, SV, SV>(stash, stash, L, P, env0, warp, lane);
    }
    const int row = tid >> 2, k = tid & 3;
    float v = 0.f;
    if (A.n_vf > 0) {                                     // the last vf layer, streamed into value_net
        const Layer& L = A.vf[A.n_vf - 1];
        if (DCP_WIDE) head_layer<2, 4, X3, 1, SV>(stash, red, L, P, A.value_w, warp, lane);
        else head_layer<1, 8, X3, 1, SV>(stash, red, L, P, A.value_w, warp, lane);
        __syncthreads();
        if (row < BM) {
            v = __ldg(P.fp + A.value_b);
            const int n_units = L.N / UNIT;
            for (int c = 0; c < n_units; ++c) v += red[c * BM + row];              // fixed order
        }
    } else if (row < BM) {                                // vf == (): value_net reads the features; the quad splits the columns
        const int F = P.layers[FINAL_LAYER].N;
        const float* w = P.fp + A.value_w;
        const float* x = stash + row * SV;
        for (int c = k; c < F; c += 4) v = fmaf(x[c], __ldg(w + c), v);
        v += __shfl_xor_sync(0xffffffffu, v, 1);
        v += __shfl_xor_sync(0xffffffffu, v, 2);
        v += __ldg(P.fp + A.value_b);
    }
    return v;
}

// tid = threadIdx.x, read by the kernel itself: there it carries the range of __launch_bounds__ (the code of policy_kernel is
// what it was before the actor-critic mode, instruction for instruction)
template <bool X3, bool AC>
__device__ __forceinline__ void policy_body(const Params& P, const ACParams* A, const int tid) {
    extern __shared__ __align__(16) float smem[];
    float* act = smem;
    float* red = smem + BM * S;
    const int warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
    const long long env0 = (long long)blockIdx.x * BM;
    const long long E = P.n_envs;

    // ---- conv1: rows (patch, env), 12 patches (2 x 6) of C x 4 x 4, K = 16 C, N = 32; h1 -> act[env][patch*32 + channel]
    {
        const int KS = 2 * P.C;                          // <= 6
        const size_t env_stride = (size_t)P.C * 338;
        const float2* wh = P.w_hi + P.conv1_w;
        const float2* wl = P.w_lo + P.conv1_w;
        for (int pass = 0; pass < 3; ++pass) {
            const int mti = warp * 3 + pass;             // m-tile: 16 envs of one patch
            const int patch = mti >> 2, py = patch / 6, px = patch % 6, el = (mti & 3) * 16 + g;
            float a[6][4];
            {
                const long long ea = env0 + el, eb = ea + 8;
                const float* pa = P.lidar + (size_t)ea * env_stride;
                const float* pb = P.lidar + (size_t)eb * env_stride;
#pragma unroll
                for (int ks = 0; ks < 6; ++ks) {
                    const int off = ((ks >> 1) * 13 + 4 * py + (ks & 1) * 2) * 26 + 4 * px + t;      // channel ks/2, row ky, column kx = t
                    const bool on = ks < KS;
                    a[ks][0] = (on && ea < E) ? __ldg(pa + off) : 0.f;
                    a[ks][1] = (on && eb < E) ? __ldg(pb + off) : 0.f;
                    a[ks][2] = (on && ea < E) ? __ldg(pa + off + 26) : 0.f;                           // k + 4: next row of the patch
                    a[ks][3] = (on && eb < E) ? __ldg(pb + off + 26) : 0.f;
                }
            }
            float acc[4][4];
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
                for (int i = 0; i < 4; ++i) acc[j][i] = 0.f;
#pragma unroll
            for (int ks = 0; ks < 6; ++ks) {
                if (ks < KS) {
                    uint32_t ah[4], al[4];
                    split_a<X3>(a[ks], ah, al);
                    float2 bh[4], bl[4];
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        bh[j] = __ldg(wh + (ks * 4 + j) * 32 + lane);
                        bl[j] = X3 ? __ldg(wl + (ks * 4 + j) * 32 + lane) : make_float2(0.f, 0.f);
                    }
                    if (X3) {
#pragma unroll
                        for (int j = 0; j < 4; ++j) mma_tf32(acc[j], al, bh[j].x, bh[j].y);
#pragma unroll
                        for (int j = 0; j < 4; ++j) mma_tf32(acc[j], ah, bl[j].x, bl[j].y);
                    }
#pragma unroll
                    for (int j = 0; j < 4; ++j) mma_tf32(acc[j], ah, bh[j].x, bh[j].y);
                }
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int col = j * 8 + 2 * t;
                const float b0 = __ldg(P.fp + P.conv1_b + col), b1 = __ldg(P.fp + P.conv1_b + col + 1);
                float* o = act + el * S + patch * 32 + col;
                *reinterpret_cast<float2*>(o) = make_float2(activate<X3>(acc[j][0] + b0, ACT_RELU), activate<X3>(acc[j][1] + b1, ACT_RELU));
                *reinterpret_cast<float2*>(o + 8 * S) = make_float2(activate<X3>(acc[j][2] + b0, ACT_RELU), activate<X3>(acc[j][3] + b1, ACT_RELU));
            }
        }
    }
    __syncthreads();

    // ---- conv2: rows (w, env), w = 0..2; K = 128 ordered (ky, kx, channel); N = 64; feature (n, w) -> act[env][n*3 + w]
    {
        const int qn = warp & 3, mg = warp >> 2;         // n-tiles qn*2, qn*2+1; m-tiles mg*3 .. +2
        float acc[3][2][4];
#pragma unroll
        for (int mt = 0; mt < 3; ++mt)
#pragma unroll
            for (int j = 0; j < 2; ++j)
#pragma unroll
                for (int i = 0; i < 4; ++i) acc[mt][j][i] = 0.f;
        mma_block<3, 2, 4, X3>(acc, [&](int mt, int ks, float (&a)[4]) {
            const int mtile = mg * 3 + mt, wpos = mtile >> 2, el = (mtile & 3) * 16 + g;
            const int q = ks >> 2, ky = q >> 1, kx = q & 1, c = (ks & 3) * 8 + t;
            const float* p = act + el * S + (ky * 6 + 2 * wpos + kx) * 32 + c;
            a[0] = p[0]; a[1] = p[8 * S]; a[2] = p[4]; a[3] = p[8 * S + 4];
        }, 16, P.w_hi + P.conv2_w, P.w_lo + P.conv2_w, qn * 2, lane);
        __syncthreads();
#pragma unroll
        for (int mt = 0; mt < 3; ++mt) {
            const int mtile = mg * 3 + mt, wpos = mtile >> 2, el = (mtile & 3) * 16 + g;
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const int n = (qn * 2 + j) * 8 + 2 * t;
                const float b0 = __ldg(P.fp + P.conv2_b + n), b1 = __ldg(P.fp + P.conv2_b + n + 1);
                float* o = act + el * S + n * 3 + wpos;
                o[0] = activate<X3>(acc[mt][j][0] + b0, ACT_RELU);
                o[3] = activate<X3>(acc[mt][j][1] + b1, ACT_RELU);
                o[8 * S] = activate<X3>(acc[mt][j][2] + b0, ACT_RELU);
                o[8 * S + 3] = activate<X3>(acc[mt][j][3] + b1, ACT_RELU);
            }
        }
        __syncthreads();
    }

    // ---- the two input MLPs, final_layer, the hidden layers of pi but the last
    for (int li = 0; li + 1 < P.n_layers; ++li) {
        const Layer& L = P.layers[li];
        if (L.N == 128 || L.N == 64) dense_layer<1, 4, X3>(act, act, L, P, env0, warp, lane);
        else if (DCP_WIDE) dense_layer<2, 4, X3>(act, act, L, P, env0, warp, lane);
        else dense_layer<1, 8, X3>(act, act, L, P, env0, warp, lane);
        if constexpr (AC) {
            // keep the features for the value branch: the next layer overwrites act only after its first barrier
            if (li == FINAL_LAYER) {
                float* stash = red + MAX_UNITS * BM * 4;
                const int q = L.N / 4;
                for (int i = tid; i < BM * q; i += THREADS)
                    reinterpret_cast<float4*>(stash + (i / q) * SV)[i % q] = reinterpret_cast<const float4*>(act + (i / q) * S)[i % q];
            }
        }
    }

    // ---- the last hidden layer, streamed into action_net
    {
        const Layer& L = P.layers[P.n_layers - 1];
        constexpr int UNIT = DCP_WIDE ? 32 : 64;         // columns per partial sum
        if (DCP_WIDE) head_layer<2, 4, X3>(act, red, L, P, P.head_w, warp, lane);
        else head_layer<1, 8, X3>(act, red, L, P, P.head_w, warp, lane);
        __syncthreads();
        const int row = tid >> 2, k = tid & 3;
        const long long env = env0 + row;
        if constexpr (!AC) {
            if (row < BM && env < E) {
                float v = __ldg(P.fp + P.head_b + k);
                const int n_units = L.N / UNIT;
                for (int c = 0; c < n_units; ++c) v += red[(c * BM + row) * 4 + k];      // fixed order: the same bits every run
                P.actions[env * 4 + k] = fminf(fmaxf(v, P.low[k]), P.high[k]);
            }
        } else {
            float mean = 0.f;                             // the Gaussian's mean: action_net's output, unclipped
            if (row < BM) {
                mean = __ldg(P.fp + P.head_b + k);
                const int n_units = L.N / UNIT;
                for (int c = 0; c < n_units; ++c) mean += red[(c * BM + row) * 4 + k];
            }
            __syncthreads();                              // red is free for the value head
            const float value = value_branch<X3>(act, red + MAX_UNITS * BM * 4, red, P, *A, env0, tid, warp, lane);
            if (row < BM) {                               // warps 0-7 whole: the shuffles below see every lane
                float a = mean;
                if (A->sample) {
                    // eps_k: Box-Muller on one Philox block (oracle/policy_ac_fragment_model.py policy_normals): k = 0, 1 take
                    // words (x, y), k = 2, 3 words (z, w); u1 = (m + 1) / 2^24 in (0, 1], angle 2 pi u2 = pi * m2 / 2^23
                    const uint4 x = dc::philox4x32_10(A->counter, (uint32_t)dc::STREAM_POLICY, A->env_offset + (uint32_t)env, 0u, A->k0, A->k1);
                    const uint32_t wr = k < 2 ? x.x : x.z, wa = k < 2 ? x.y : x.w;
                    const float r = sqrtf(-2.f * logf((float)((wr >> 8) + 1u) * (1.f / 16777216.f)));
                    float sn, cs;
                    sincospif((float)(wa >> 8) * (1.f / 8388608.f), &sn, &cs);
                    const float eps = r * ((k & 1) ? sn : cs);
                    const float log_std = __ldg(P.fp + A->log_std + k);
                    a = fmaf(expf(log_std), eps, mean);
                    float lp = fmaf(-0.5f * eps, eps, -log_std);
                    lp += __shfl_xor_sync(0xffffffffu, lp, 1);    // (k0 + k1) + (k2 + k3) on every lane of the quad
                    lp += __shfl_xor_sync(0xffffffffu, lp, 2);
                    if (env < E) {
                        A->raw[env * 4 + k] = a;
                        if (k == 0) A->log_prob[env] = lp - 3.6757541328186907f;  // - 4 * 0.5 * log(2 pi)
                    }
                }
                if (env < E) {
                    P.actions[env * 4 + k] = fminf(fmaxf(a, P.low[k]), P.high[k]);
                    if (k == 0) A->value[env] = value;
                }
            }
        }
    }
}

template <bool X3>
__global__ void __launch_bounds__(THREADS, 1) policy_kernel(const __grid_constant__ Params P) {
    policy_body<X3, false>(P, nullptr, threadIdx.x);
}

template <bool X3>
__global__ void __launch_bounds__(THREADS, 1) policy_ac_kernel(const __grid_constant__ ACParams A) {
    policy_body<X3, true>(A.p, &A, threadIdx.x);
}

// Weights [N][K] (torch layout) -> B fragments in consumption order, split into a TF32 head and tail.
// kmap 0: k is the flat input index (zero-padded to a multiple of 8); kmap 1: conv2, k = (ky*2 + kx)*32 + c reads
// W[n][c][ky][kx].
__global__ void pack_kernel(const float* __restrict__ W, int N, int K, int KS, int kmap, int ntg, float2* __restrict__ hi, float2* __restrict__ lo) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    const int total = (N >> 3) * KS * 32;
    if (idx >= total) return;
    // order: [group of ntg n-tiles][k-step][n-tile in group][lane]
    const int lane = idx & 31, j = (idx >> 5) % ntg, ks = ((idx >> 5) / ntg) % KS, nt = ((idx >> 5) / (ntg * KS)) * ntg + j;
    const int g = lane >> 2, t = lane & 3, n = nt * 8 + g;
    float w[2];
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        const int k = ks * 8 + t + 4 * i;
        if (kmap == 1) w[i] = W[(size_t)n * K + (k & 31) * 4 + (k >> 5)];
        else w[i] = k < K ? W[(size_t)n * K + k] : 0.f;
    }
    const float h0 = __uint_as_float(tf32_rna(w[0])), h1 = __uint_as_float(tf32_rna(w[1]));
    hi[idx] = make_float2(h0, h1);
    lo[idx] = make_float2(w[0] - h0, w[1] - h1);
}

}  // namespace dcp

struct dc_policy {
    int device = 0;
    dcp::Params p{};
    bool ac = false;                 // made by dc_policy_create_ac: `a` holds the value branch (a.p == p)
    dcp::ACParams a{};
    float2* w_hi = nullptr;
    float2* w_lo = nullptr;
    float* fp = nullptr;
};

namespace {

int pfail(int code, const std::string& msg) { dc_internal_set_error(msg.c_str()); return code; }
#define DCP_CUDA(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return pfail(DC_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__)); } while (0)

struct PackJob { const float* W; int N, K, KS, kmap, ntg, w_off; };

// widths the fused kernel holds: an intermediate layer is one pass of 8 warps (<= 256 columns, multiples of 64); the last
// hidden layer streams through the head in chunks of 64 columns
bool widths_ok(const std::vector<int>& widths) {
    for (size_t i = 0; i < widths.size(); ++i) {
        const bool last = i + 1 == widths.size();
        const int n = widths[i];
        if (n < 64 || n % 64 || n > (last ? 64 * dcp::MAX_CHUNKS : 256)) return false;
    }
    return true;
}

// dc_policy_create (v == nullptr) and dc_policy_create_ac
int create(const dc_policy_weights* w, const dc_value_weights* v, int device, dc_policy** out, const char* who) {
    using namespace dcp;
    const std::string fn(who);
    if (!w || !out) return pfail(DC_ERR_ARG, fn + ": null argument");
    *out = nullptr;
    const int C = w->lidar_channels, F = w->features_dim, n_pi = w->n_pi;
    if (C < 1 || C > 3) return pfail(DC_ERR_ARG, fn + ": lidar_channels must be 1..3");
    if (n_pi < 0 || n_pi > 8) return pfail(DC_ERR_ARG, fn + ": n_pi must be 0..8");
    if (w->activation != ACT_RELU && w->activation != ACT_TANH) return pfail(DC_ERR_ARG, fn + ": activation must be 1 (ReLU) or 2 (Tanh)");
    std::vector<int> widths{F};
    for (int i = 0; i < n_pi; ++i) widths.push_back(w->pi[i]);
    if (!widths_ok(widths))
        return pfail(DC_ERR_ARG, fn + ": features_dim and the hidden widths of pi must be multiples of 64, at most 256 "
                                      "(the last one at most 1024); use the torch module for other shapes");
    const float* need[] = {w->conv1_w, w->conv1_b, w->conv2_w, w->conv2_b, w->final_w, w->final_b, w->head_w, w->head_b};
    for (const float* p : need) if (!p) return pfail(DC_ERR_ARG, fn + ": null weight pointer");
    for (int i = 0; i < 3; ++i)
        if (!w->inertial_w[i] || !w->inertial_b[i] || !w->action_w[i] || !w->action_b[i]) return pfail(DC_ERR_ARG, fn + ": null MLP weight pointer");
    for (int i = 0; i < n_pi; ++i) if (!w->pi_w[i] || !w->pi_b[i]) return pfail(DC_ERR_ARG, fn + ": null pi weight pointer");
    if (v) {
        if (v->n_vf < 0 || v->n_vf > MAX_VF) return pfail(DC_ERR_ARG, fn + ": n_vf must be 0..8");
        std::vector<int> vw{F};
        for (int i = 0; i < v->n_vf; ++i) vw.push_back(v->vf[i]);
        if (F > SV - 4 || !widths_ok(vw))
            return pfail(DC_ERR_ARG, fn + ": the hidden widths of vf must be multiples of 64, at most 256 (the last one at most 1024)");
        for (int i = 0; i < v->n_vf; ++i) if (!v->vf_w[i] || !v->vf_b[i]) return pfail(DC_ERR_ARG, fn + ": null vf weight pointer");
        if (!v->value_w || !v->value_b || !v->log_std) return pfail(DC_ERR_ARG, fn + ": null value_net / log_std pointer");
    }
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0) { cudaGetLastError(); return pfail(DC_ERR_NO_DEVICE, fn + ": no CUDA device (there is no CPU fallback)"); }
    DCP_CUDA(cudaSetDevice(device));

    dc_policy* P = new (std::nothrow) dc_policy;
    if (!P) return pfail(DC_ERR_ARG, fn + ": out of host memory");
    P->device = device;
    Params& p = P->p;
    p.C = C;
    std::vector<PackJob> jobs;
    struct BiasJob { const float* src; int n, off; };
    std::vector<BiasJob> biases;
    int w_total = 0, f_total = 0;
    auto add_w = [&](const float* W, int N, int K, int kmap, int ntg) {
        const int KS = (K + 7) / 8, off = w_total;
        jobs.push_back({W, N, K, KS, kmap, ntg, off});
        w_total += (N / 8) * KS * 32;
        return off;
    };
    auto add_f = [&](const float* src, int n) { const int off = f_total; biases.push_back({src, n, off}); f_total += (n + 3) & ~3; return off; };
    p.conv1_w = add_w(w->conv1_w, 32, 16 * C, 0, 4); p.conv1_b = add_f(w->conv1_b, 32);
    p.conv2_w = add_w(w->conv2_w, 64, 128, 1, 4);    p.conv2_b = add_f(w->conv2_b, 64);
    auto make_layer = [&](const float* W, const float* b, int K, int N, int in_off, int out_off, int act, int src) {
        Layer L;
        L.K = K; L.KS = (K + 7) / 8; L.N = N; L.in_off = in_off; L.out_off = out_off; L.act = act; L.src = src;
        L.w_off = add_w(W, N, K, 0, 8); L.b_off = add_f(b, N);
        return L;
    };
    int nl = 0;
    auto add_layer = [&](const float* W, const float* b, int K, int N, int in_off, int out_off, int act, int src) {
        p.layers[nl++] = make_layer(W, b, K, N, in_off, out_off, act, src);
    };
    add_layer(w->inertial_w[0], w->inertial_b[0], 15, 128, 0, 192, ACT_RELU, SRC_INERTIAL);
    add_layer(w->inertial_w[1], w->inertial_b[1], 128, 128, 192, 192, ACT_RELU, SRC_SMEM);
    add_layer(w->inertial_w[2], w->inertial_b[2], 128, 128, 192, 192, ACT_RELU, SRC_SMEM);
    add_layer(w->action_w[0], w->action_b[0], 4, 128, 0, 320, ACT_RELU, SRC_ACTION);
    add_layer(w->action_w[1], w->action_b[1], 128, 128, 320, 320, ACT_RELU, SRC_SMEM);
    add_layer(w->action_w[2], w->action_b[2], 128, 128, 320, 320, ACT_RELU, SRC_SMEM);
    add_layer(w->final_w, w->final_b, 448, F, 0, 0, ACT_RELU, SRC_SMEM);      // FINAL_LAYER
    int width = F;
    for (int i = 0; i < n_pi; ++i) {
        add_layer(w->pi_w[i], w->pi_b[i], width, w->pi[i], 0, 0, w->activation, SRC_SMEM);
        width = w->pi[i];
    }
    p.n_layers = nl;
    p.head_w = add_f(w->head_w, 4 * width);
    p.head_b = add_f(w->head_b, 4);
    for (int k = 0; k < 4; ++k) { p.low[k] = w->low[k]; p.high[k] = w->high[k]; }
    if (v) {
        ACParams& a = P->a;
        P->ac = true;
        a.n_vf = v->n_vf;
        int vw = F;
        for (int i = 0; i < v->n_vf; ++i) {                                    // in place in the stash
            a.vf[i] = make_layer(v->vf_w[i], v->vf_b[i], vw, v->vf[i], 0, 0, w->activation, SRC_SMEM);
            vw = v->vf[i];
        }
        a.value_w = add_f(v->value_w, vw);
        a.value_b = add_f(v->value_b, 1);
        a.log_std = add_f(v->log_std, 4);
    }

    auto cleanup = [&]() { cudaFree(P->w_hi); cudaFree(P->w_lo); cudaFree(P->fp); delete P; };
    cudaError_t e;
    const size_t w_alloc = sizeof(float2) * ((size_t)w_total + PAD_STEPS * 8 * 32);
    if ((e = cudaMalloc(&P->w_hi, w_alloc)) != cudaSuccess || (e = cudaMalloc(&P->w_lo, w_alloc)) != cudaSuccess ||
        (e = cudaMalloc(&P->fp, sizeof(float) * (size_t)f_total)) != cudaSuccess) {
        cleanup();
        return pfail(DC_ERR_CUDA, fn + ": cudaMalloc: " + cudaGetErrorString(e));
    }
    if ((e = cudaMemset(P->w_hi, 0, w_alloc)) != cudaSuccess || (e = cudaMemset(P->w_lo, 0, w_alloc)) != cudaSuccess ||
        (e = cudaMemset(P->fp, 0, sizeof(float) * (size_t)f_total)) != cudaSuccess) { cleanup(); return pfail(DC_ERR_CUDA, fn + ": cudaMemset"); }
    for (const PackJob& j : jobs) {
        const int total = (j.N / 8) * j.KS * 32;
        pack_kernel<<<(total + 255) / 256, 256>>>(j.W, j.N, j.K, j.KS, j.kmap, j.ntg, P->w_hi + j.w_off, P->w_lo + j.w_off);
        dc_internal_count_launches(1);
    }
    for (const BiasJob& b : biases)
        if ((e = cudaMemcpy(P->fp + b.off, b.src, sizeof(float) * (size_t)b.n, cudaMemcpyDefault)) != cudaSuccess) {
            cleanup();
            return pfail(DC_ERR_CUDA, fn + ": cudaMemcpy of a bias / head tensor: " + cudaGetErrorString(e));
        }
    if ((e = cudaDeviceSynchronize()) != cudaSuccess || (e = cudaGetLastError()) != cudaSuccess) {
        cleanup();
        return pfail(DC_ERR_CUDA, fn + ": packing the weights: " + cudaGetErrorString(e));
    }
    p.w_hi = P->w_hi; p.w_lo = P->w_lo; p.fp = P->fp;
    P->a.p = p;
    if ((e = cudaFuncSetAttribute(policy_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES)) != cudaSuccess ||
        (e = cudaFuncSetAttribute(policy_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES)) != cudaSuccess ||
        (v && (e = cudaFuncSetAttribute(policy_ac_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_AC_BYTES)) != cudaSuccess) ||
        (v && (e = cudaFuncSetAttribute(policy_ac_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_AC_BYTES)) != cudaSuccess)) {
        cleanup();
        return pfail(DC_ERR_CUDA, fn + ": cudaFuncSetAttribute: " + cudaGetErrorString(e));
    }
    *out = P;
    return DC_OK;
}

}  // namespace

extern "C" {

int dc_policy_create(const dc_policy_weights* w, int device, dc_policy** out) {
    return create(w, nullptr, device, out, "dc_policy_create");
}

int dc_policy_create_ac(const dc_policy_weights* w, const dc_value_weights* v, int device, dc_policy** out) {
    if (!v) return pfail(DC_ERR_ARG, "dc_policy_create_ac: null argument");
    return create(w, v, device, out, "dc_policy_create_ac");
}

int dc_policy_forward(dc_policy* P, const float* lidar, const float* inertial, const float* last_action, int64_t n_envs,
                      float* actions, int32_t precision, void* stream) {
    using namespace dcp;
    if (!P || !lidar || !inertial || !last_action || !actions || n_envs < 0) return pfail(DC_ERR_ARG, "dc_policy_forward: bad argument");
    if (precision != 0 && precision != 1) return pfail(DC_ERR_ARG, "dc_policy_forward: precision must be 0 (3 x TF32, float32-grade) or 1 (TF32)");
    if (n_envs == 0) return DC_OK;
    const long long blocks = (n_envs + BM - 1) / BM;
    if (blocks > 0x7fffffffLL) return pfail(DC_ERR_ARG, "dc_policy_forward: too many envs for one launch");
    Params p = P->p;
    p.lidar = lidar; p.inertial = inertial; p.last_action = last_action; p.actions = actions; p.n_envs = n_envs;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (precision == 0) policy_kernel<true><<<(unsigned)blocks, THREADS, SMEM_BYTES, st>>>(p);
    else policy_kernel<false><<<(unsigned)blocks, THREADS, SMEM_BYTES, st>>>(p);
    dc_internal_count_launches(1);
    DCP_CUDA(cudaGetLastError());
    return DC_OK;
}

int dc_policy_act(dc_policy* P, const float* lidar, const float* inertial, const float* last_action, int64_t n_envs,
                  uint64_t seed, int64_t env_offset, uint32_t counter, int32_t sample, float* env_actions, float* raw_actions,
                  float* log_prob, float* value, int32_t precision, void* stream) {
    using namespace dcp;
    if (!P || !lidar || !inertial || !last_action || !env_actions || !value || n_envs < 0) return pfail(DC_ERR_ARG, "dc_policy_act: bad argument");
    if (!P->ac) return pfail(DC_ERR_ARG, "dc_policy_act: the policy was made by dc_policy_create, without a value branch (use dc_policy_create_ac)");
    if (sample != 0 && sample != 1) return pfail(DC_ERR_ARG, "dc_policy_act: sample must be 0 (mean action) or 1");
    if (sample && (!raw_actions || !log_prob)) return pfail(DC_ERR_ARG, "dc_policy_act: sample = 1 needs raw_actions and log_prob");
    if (precision != 0 && precision != 1) return pfail(DC_ERR_ARG, "dc_policy_act: precision must be 0 (3 x TF32, float32-grade) or 1 (TF32)");
    if (env_offset < 0 || env_offset + n_envs > (1LL << 32)) return pfail(DC_ERR_ARG, "dc_policy_act: env_offset + n_envs must lie in [0, 2^32]");
    if (n_envs == 0) return DC_OK;
    const long long blocks = (n_envs + BM - 1) / BM;
    if (blocks > 0x7fffffffLL) return pfail(DC_ERR_ARG, "dc_policy_act: too many envs for one launch");
    ACParams a = P->a;
    a.p.lidar = lidar; a.p.inertial = inertial; a.p.last_action = last_action; a.p.actions = env_actions; a.p.n_envs = n_envs;
    a.raw = raw_actions; a.log_prob = log_prob; a.value = value;
    a.k0 = (uint32_t)seed; a.k1 = (uint32_t)(seed >> 32); a.env_offset = (uint32_t)env_offset; a.counter = counter; a.sample = sample;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (precision == 0) policy_ac_kernel<true><<<(unsigned)blocks, THREADS, SMEM_AC_BYTES, st>>>(a);
    else policy_ac_kernel<false><<<(unsigned)blocks, THREADS, SMEM_AC_BYTES, st>>>(a);
    dc_internal_count_launches(1);
    DCP_CUDA(cudaGetLastError());
    return DC_OK;
}

void dc_policy_destroy(dc_policy* P) {
    if (!P) return;
    cudaFree(P->w_hi); cudaFree(P->w_lo); cudaFree(P->fp);
    delete P;
}

}  // extern "C"

// Shared helpers for libddrl_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/ddrl_b200.h"

namespace ddrl {

void set_error(const char* fmt, ...);
void count_launch(int n = 1);

#define DDRL_REQUIRE(cond, code, ...)            \
    do {                                          \
        if (!(cond)) {                            \
            ::ddrl::set_error(__VA_ARGS__);       \
            return (code);                        \
        }                                         \
    } while (0)

#define DDRL_CHECK_LAUNCH(name)                                                        \
    do {                                                                               \
        cudaError_t e__ = cudaGetLastError();                                          \
        if (e__ != cudaSuccess) {                                                      \
            ::ddrl::set_error("%s: launch failed: %s", name, cudaGetErrorString(e__)); \
            return DDRL_E_CUDA;                                                        \
        }                                                                              \
        ::ddrl::count_launch();                                                        \
    } while (0)

// Raises the dynamic shared-memory limit of kernel Kern to 227 KB (the sm_100a opt-in maximum) before its first launch;
// the flag is a static of each instantiation, i.e. one per kernel.
template <auto Kern>
inline int raise_smem_once(const char* who) {
    static bool done = false;
    if (!done) {
        if (cudaFuncSetAttribute(Kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024) != cudaSuccess) {
            set_error("%s: cannot raise dynamic shared memory: %s", who, cudaGetErrorString(cudaGetLastError()));
            return DDRL_E_CUDA;
        }
        done = true;
    }
    return DDRL_OK;
}

// FCNet flat-parameter offsets (checkpoint order, include/ddrl_b200.h).
struct FcOffsets {
    int W1, b1, Wv1, bv1, W2, b2, Wv2, bv2, Wo, bo, Wvo, bvo, NP;
};
__host__ __device__ inline FcOffsets fc_offsets(int D, int A) {
    FcOffsets o;
    const int H = DDRL_HIDDEN;
    int p = 0;
    o.W1 = p;  p += D * H;
    o.b1 = p;  p += H;
    o.Wv1 = p; p += D * H;
    o.bv1 = p; p += H;
    o.W2 = p;  p += H * H;
    o.b2 = p;  p += H;
    o.Wv2 = p; p += H * H;
    o.bv2 = p; p += H;
    o.Wo = p;  p += H * 2 * A;
    o.bo = p;  p += 2 * A;
    o.Wvo = p; p += H;
    o.bvo = p; p += 1;
    o.NP = p;
    return o;
}

constexpr float kLog2Pi = 1.8378770664093453f;

// RLlib DiagGaussian (models/tf/tf_action_dist.py) sample of row r: action[r][i] = mean + exp(log_std) * eps[r][i] for
// logits[r] = (mean | log_std) [2A]; returns logp(action) = -0.5 sum z^2 - 0.5 log(2 pi) A - sum log_std,
// z = (action - mean) / exp(log_std), summed in the order i = 0..A-1.  dg_sample_kernel and graphnet_fwd_warp_kernel<true>
// both call it, so their actions and logp are bit-identical.
__device__ __forceinline__ float dg_sample_row(const float* __restrict__ logits, const float* __restrict__ eps, int64_t r,
                                               int A, float* __restrict__ action) {
    float sz2 = 0.f, sls = 0.f;
    for (int i = 0; i < A; ++i) {
        const float mu = logits[r * 2 * A + i], ls = logits[r * 2 * A + A + i];
        const float sd = expf(ls);
        const float a = mu + sd * eps[r * A + i];
        const float z = (a - mu) / sd;
        sz2 = fmaf(z, z, sz2);
        sls += ls;
        action[r * A + i] = a;
    }
    return -0.5f * sz2 - 0.5f * kLog2Pi * (float)A - sls;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

}  // namespace ddrl

// Shared pieces of the tensor-core (tcgen05) FCNet training kernels: launch arguments, operand scales, the split-fp16
// GEMM issue loop and the fp32 <-> (hi, lo) fp16 converters.  See the header comment of the kernel in tc.cu.
#pragma once
#include <cuda_fp16.h>

#include <type_traits>

#include "common.cuh"
#include "fcnet_tc_layout.cuh"
#include "ppo_loss.cuh"
#include "sgd_tail.cuh"
#include "umma.cuh"

namespace ddrl {

struct TcTrainArgs {
    const unsigned char* img;
    const float *obs, *actions, *old_logits, *old_logp, *vf_preds, *adv, *vtarg;
    int64_t R;
    int D, A, MB;
    const int32_t* mb_perm;
    int64_t perm_stride;
    const int32_t* step_ctr;
    const float* kl_coeff;
    ddrl_ppo_hyper hp;
    float* grad_part;
    double* stat_part;
    int* status;
    long long* dbg_clock;   // optional: CTA (0, 0) thread 0 stores clock64() at phase boundaries (ddrl_tc_set_debug_clock)
    SgdTail tail;
    // forward-only mode of the ping-pong kernel (inference: ddrl_fcnet_forward_tc): filter table, outputs, sampling noise
    const double* norm;     // [P][2][D] mean, 1/(std + 1e-8) or nullptr
    float clip;
    float *obs_out, *logits_out, *value_out, *action_out, *logp_out;
    const float* eps;
};

// ping-pong variant (tc2.cu); A in {1,2,4,8}, tc2_eligible(D, A): D <= 47
int launch_tc2(const TcTrainArgs& a, int P, int G, cudaStream_t st);
int launch_tc2_forward(const TcTrainArgs& a, int P, int G, cudaStream_t st);
// leg-coupled ping-pong step (SharedDecentralLegID): A = 2, D in {19, 20}; node_id [P][R], theta [P][NP + 8]
int launch_tc2_cup(const TcTrainArgs& a, const int32_t* node_id, const float* theta, int P, int G, cudaStream_t st);
// leg-coupled inference forward (P = 1, A = 2, tc2_eligible D): node_id [R], coupling [4][2]
int launch_tc2_forward_cup(const TcTrainArgs& a, const int32_t* node_id, const float* coupling, int G, cudaStream_t st);
// true if ddrl_tc_set_cluster asked for thread-block clusters on the ping-pong step
bool tc2_clusters_requested();

// launch(std::integral_constant<int, A>) for the action widths the tensor-core kernels are instantiated for, A in {1,2,4,8}
template <class Launch>
int dispatch_A(int A, const char* unsupported, Launch&& launch) {
    switch (A) {
        case 1: return launch(std::integral_constant<int, 1>{});
        case 2: return launch(std::integral_constant<int, 2>{});
        case 4: return launch(std::integral_constant<int, 4>{});
        case 8: return launch(std::integral_constant<int, 8>{});
        default: set_error("%s", unsupported); return DDRL_E_UNSUPPORTED_SHAPE;
    }
}

// Power-of-two operand scales (see header comment).  What matters is the absolute error relative to the tensor's
// scale: entries too small for a normal lo half lose at most 2^-25/scale, negligible next to the entries that dominate.
constexpr float TC_SX = 16.f;      // observations (|x| <= 3750)
constexpr float TC_SH = 4096.f;    // tanh activations (|h| <= 1)
constexpr float TC_SW = 256.f;     // weights (|w| <= 234)
// Loss gradients (dl and the dz2 / dz1 derived from it) have no a-priori scale (it follows |v - R| and the
// advantages), so each branch picks ONE power-of-two scale per CTA from the first tile: max|dl| * scale ~ 256, which
// leaves a factor 234 of headroom for |dz| to exceed |dl| before the fp16 range is hit (then: flagged, never silent).
constexpr float TC_GTARGET = 256.f;

__device__ __forceinline__ void tc_cp16(unsigned char* smem_dst, const unsigned char* gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(umma::smem_u32(smem_dst)), "l"(gsrc));
}
__device__ __forceinline__ void tc_cp4(float* smem_dst, const float* gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(umma::smem_u32(smem_dst)), "l"(gsrc));
}

// D[tmem] (+)= A * B^T with fp16 (hi, lo) operands: products (hi,hi) (hi,lo) (lo,hi); nprod == 2 -> (hi,hi) (lo,hi).
// a_rows / b_rows = row count of the chunked buffers; *_mn selects the MN-major view.  One thread calls this.
__device__ __forceinline__ void tc_gemm(uint32_t d_tmem, uint32_t a_hi, uint32_t a_lo, int a_rows, bool a_mn, uint32_t b_hi,
                                        uint32_t b_lo, int b_rows, bool b_mn, int M, int N, int nk, bool accumulate, int nprod) {
    const uint32_t idesc = umma::idesc_f16(M, N, a_mn, b_mn);
    // descriptors advance along K by adding to the 14-bit start-address field (16-byte units; smem < 256 KB, no carry)
    const uint64_t astep = a_mn ? 16u : (uint64_t)(2 * a_rows);
    const uint64_t bstep = b_mn ? 16u : (uint64_t)(2 * b_rows);
    const uint64_t ah = a_mn ? umma::desc_mnmajor(a_hi, a_rows) : umma::desc_kmajor(a_hi, a_rows);
    const uint64_t al = a_mn ? umma::desc_mnmajor(a_lo, a_rows) : umma::desc_kmajor(a_lo, a_rows);
    const uint64_t bh = b_mn ? umma::desc_mnmajor(b_hi, b_rows) : umma::desc_kmajor(b_hi, b_rows);
    const uint64_t bl = b_mn ? umma::desc_mnmajor(b_lo, b_rows) : umma::desc_kmajor(b_lo, b_rows);
    uint32_t acc = accumulate ? 1u : 0u;
#pragma unroll 1
    for (int pr = 0; pr < nprod; ++pr) {
        uint64_t ad = (pr == 2 || (nprod == 2 && pr == 1)) ? al : ah;
        uint64_t bd = (nprod == 3 && pr == 1) ? bl : bh;
#pragma unroll 4
        for (int ks = 0; ks < nk; ++ks) {
            umma::mma_f16(d_tmem, ad, bd, idesc, acc != 0u);
            acc = 1u;
            ad += astep;
            bd += bstep;
        }
    }
}

// Same with an explicit product mask (bit 0: hi*hi, bit 1: hi*lo, bit 2: lo*hi): lets several issuing warps share one
// GEMM by product, each into its own accumulator (the accumulators are added at read-out).
__device__ __forceinline__ void tc_gemm_mask(uint32_t d_tmem, uint32_t a_hi, uint32_t a_lo, int a_rows, bool a_mn, uint32_t b_hi,
                                             uint32_t b_lo, int b_rows, bool b_mn, int M, int N, int nk, bool accumulate, int pmask) {
    const uint32_t idesc = umma::idesc_f16(M, N, a_mn, b_mn);
    const uint64_t astep = a_mn ? 16u : (uint64_t)(2 * a_rows);
    const uint64_t bstep = b_mn ? 16u : (uint64_t)(2 * b_rows);
    const uint64_t ah = a_mn ? umma::desc_mnmajor(a_hi, a_rows) : umma::desc_kmajor(a_hi, a_rows);
    const uint64_t al = a_mn ? umma::desc_mnmajor(a_lo, a_rows) : umma::desc_kmajor(a_lo, a_rows);
    const uint64_t bh = b_mn ? umma::desc_mnmajor(b_hi, b_rows) : umma::desc_kmajor(b_hi, b_rows);
    const uint64_t bl = b_mn ? umma::desc_mnmajor(b_lo, b_rows) : umma::desc_kmajor(b_lo, b_rows);
    uint32_t acc = accumulate ? 1u : 0u;
#pragma unroll 1
    for (int pr = 0; pr < 3; ++pr) {
        if (!((pmask >> pr) & 1)) continue;
        uint64_t ad = pr == 2 ? al : ah;
        uint64_t bd = pr == 1 ? bl : bh;
#pragma unroll 4
        for (int ks = 0; ks < nk; ++ks) {
            umma::mma_f16(d_tmem, ad, bd, idesc, acc != 0u);
            acc = 1u;
            ad += astep;
            bd += bstep;
        }
    }
}

#ifndef TC_MMA_UNROLL_N
#define TC_MMA_UNROLL_N 1
#endif
constexpr int TC_MMA_UNROLL = TC_MMA_UNROLL_N;   // K-step unrolling of the warp-uniform issue loops: 1 — a dependent MMA takes ~100
                                                 // cycles anyway, and 26 KB less code measured 0.5 us per step faster (i-cache)

// Warp-uniform variants: the WHOLE warp calls these with warp-uniform arguments (kernel parameters, constants,
// __shfl_sync(.., 0) results); one elected lane issues each instruction.  ptxas then keeps descriptors and TMEM addresses in
// uniform registers and emits bare UTCHMMA instructions instead of a per-instruction R2UR waterfall loop
// (profiles/r02_umma_issue_bench.txt: 148 -> 100 cycles per dependent MMA, 39-50 with independent accumulators interleaved).
__device__ __forceinline__ void tc_gemm_mask_u(uint32_t d_tmem, uint32_t a_hi, uint32_t a_lo, int a_rows, bool a_mn, uint32_t b_hi,
                                               uint32_t b_lo, int b_rows, bool b_mn, int M, int N, int nk, bool accumulate,
                                               int pmask) {
    const uint32_t idesc = umma::idesc_f16(M, N, a_mn, b_mn);
    const uint64_t astep = a_mn ? 16u : (uint64_t)(2 * a_rows);
    const uint64_t bstep = b_mn ? 16u : (uint64_t)(2 * b_rows);
    const uint64_t ah = a_mn ? umma::desc_mnmajor(a_hi, a_rows) : umma::desc_kmajor(a_hi, a_rows);
    const uint64_t al = a_mn ? umma::desc_mnmajor(a_lo, a_rows) : umma::desc_kmajor(a_lo, a_rows);
    const uint64_t bh = b_mn ? umma::desc_mnmajor(b_hi, b_rows) : umma::desc_kmajor(b_hi, b_rows);
    const uint64_t bl = b_mn ? umma::desc_mnmajor(b_lo, b_rows) : umma::desc_kmajor(b_lo, b_rows);
    uint32_t acc = accumulate ? 1u : 0u;
#pragma unroll
    for (int pr = 0; pr < 3; ++pr) {
        if (!((pmask >> pr) & 1)) continue;
        uint64_t ad = pr == 2 ? al : ah;
        uint64_t bd = pr == 1 ? bl : bh;
#pragma unroll TC_MMA_UNROLL
        for (int ks = 0; ks < nk; ++ks) {
            umma::mma_f16_elect(d_tmem, ad, bd, idesc, acc);
            acc = 1u;
            ad += astep;
            bd += bstep;
        }
    }
}
// nprod == 3: (hi,hi) (hi,lo) (lo,hi); nprod == 2: (hi,hi) (lo,hi)
__device__ __forceinline__ void tc_gemm_u(uint32_t d_tmem, uint32_t a_hi, uint32_t a_lo, int a_rows, bool a_mn, uint32_t b_hi,
                                          uint32_t b_lo, int b_rows, bool b_mn, int M, int N, int nk, bool accumulate, int nprod) {
    tc_gemm_mask_u(d_tmem, a_hi, a_lo, a_rows, a_mn, b_hi, b_lo, b_rows, b_mn, M, N, nk, accumulate, nprod == 3 ? 7 : 5);
}

// Weight-gradient GEMM with the hi | lo halves of the A operand STACKED along M (warp-uniform issue, see above):
//     D[128][N] (+)= [A_hi | A_lo]^T * B        (A, B MN-major views of chunked buffers: the reduction runs over rows)
// The lo buffer of every activation follows its hi buffer in shared memory, i.e. it continues the hi buffer's chunk sequence,
// so ONE M = 128 instruction over the 16 chunks computes A_hi^T B (accumulator rows 0-63) and A_lo^T B (rows 64-127): the
// M = 64 weight-gradient GEMMs left half of the tensor core's M idle, and their three products were three dependent MMAs per
// 16 rows of K — a dependent MMA costs ~100 cycles whatever its shape (profiles/r02_umma_issue_bench.txt), so the chain
// length, not the math, set the time of the backward stages.  B is either the hi | lo pair itself as ONE operand of 2 x cols
// columns (ngroups == 1, b1 unused: all four products from nk MMAs; the reader adds the two column blocks) or hi and lo one
// after the other into the same columns (ngroups == 2: 2 nk MMAs).  The reader adds accumulator rows m and m + 64.  The
// fourth product lo * lo (~2^-22 relative) comes for free and only moves the result closer to the FP32 product.
__device__ __forceinline__ void tc_gemm_stack_u(uint32_t d_tmem, uint32_t a_hi, int a_rows, uint32_t b0, uint32_t b1, int b_rows,
                                                int N, int nk, bool accumulate, int ngroups) {
    const uint32_t idesc = umma::idesc_f16(128, N, true, true);
    const uint64_t ad0 = umma::desc_mnmajor(a_hi, a_rows);
    uint32_t acc = accumulate ? 1u : 0u;
#pragma unroll
    for (int g = 0; g < 2; ++g) {
        if (g >= ngroups) continue;
        uint64_t ad = ad0;
        uint64_t bd = umma::desc_mnmajor(g ? b1 : b0, b_rows);
#pragma unroll TC_MMA_UNROLL
        for (int ks = 0; ks < nk; ++ks) {
            umma::mma_f16_elect(d_tmem, ad, bd, idesc, acc);
            acc = 1u;
            ad += 16u;
            bd += 16u;
        }
    }
}

// split 8 floats (times a power-of-two scale) into fp16 hi / lo 16-byte chunks; returns true on fp16 overflow
__device__ __forceinline__ bool tc_split8(const float* v, float scale, uint4& hi, uint4& lo) {
    uint32_t h[4], l[4];
    bool ovf = false;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        float x0 = v[2 * i] * scale, x1 = v[2 * i + 1] * scale;
        ovf = ovf || !(fabsf(x0) <= 60000.f) || !(fabsf(x1) <= 60000.f);
        x0 = fminf(fmaxf(x0, -60000.f), 60000.f);
        x1 = fminf(fmaxf(x1, -60000.f), 60000.f);
        const __half h0 = __float2half_rn(x0), h1 = __float2half_rn(x1);
        const __half2 hh = __halves2half2(h0, h1);
        const __half2 ll = __halves2half2(__float2half_rn(x0 - __half2float(h0)), __float2half_rn(x1 - __half2float(h1)));
        h[i] = *reinterpret_cast<const uint32_t*>(&hh);
        l[i] = *reinterpret_cast<const uint32_t*>(&ll);
    }
    hi = make_uint4(h[0], h[1], h[2], h[3]);
    lo = make_uint4(l[0], l[1], l[2], l[3]);
    return ovf;
}

// hi + lo chunk -> 8 floats (times inv_scale)
__device__ __forceinline__ void tc_join8(const uint4& hi, const uint4& lo, float inv_scale, float* v) {
    const __half2* h = reinterpret_cast<const __half2*>(&hi);
    const __half2* l = reinterpret_cast<const __half2*>(&lo);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float2 fh = __half22float2(h[i]), fl = __half22float2(l[i]);
        v[2 * i] = (fh.x + fl.x) * inv_scale;
        v[2 * i + 1] = (fh.y + fl.y) * inv_scale;
    }
}


}  // namespace ddrl

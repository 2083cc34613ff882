// FCNet (models/fcnet_glorot_uniform_init.py) grouped per-leg forward and the fused
// forward + PPO-loss + backward minibatch kernel.  FP32 FMA path ("parity mode": accurate tanhf/expf,
// fixed summation order => bit-reproducible run to run).
//
// Tiling (both kernels): a CTA of 256 threads owns the weights of ONE policy in shared memory and
// walks over 64-row tiles.  The policy and value branches have identical shapes, so they are run as
// one 128-wide network: layer 1 is x[64,D] * [W1|Wv1][D,128], layer 2 is block diagonal.  Every
// thread owns a 4-row x 8-column register tile: ty = tid/16 -> rows 4ty..4ty+3; tx = tid%16 -> branch
// tx/8 (0 policy, 1 value) and, inside the 64 columns of the branch, the two float4 groups
// [4(tx%8), +4) and [32 + 4(tx%8), +4) — so the 8 lanes of a quarter warp read 128 contiguous bytes of
// a weight row (conflict-free 128-bit shared loads; 32 FMA per 3 LDS.128).  Activations stay in shared
// memory (row-major, stride 132 floats) and are overwritten in place by their gradients on the way
// back; weight gradients accumulate in registers across all tiles of the CTA and leave as one per-CTA
// partial (reduced in fixed order by ddrl_grad_reduce => deterministic).
//
// Weights reach shared memory either from the flat checkpoint-order vector (any caller) or from a
// pre-packed "image" (exactly the shared-memory layout, maintained by ddrl_clip_adam / ddrl_fcnet_pack)
// with one straight 128-bit copy — the SGD loop uses the image so the per-step weight (re)load costs a
// coalesced 88 KB read from L2 instead of 11 K scattered loads + transposes.
#include <math.h>

#include <algorithm>

#include "common.cuh"
#include "fcnet_layout.cuh"
#include "ppo_loss.cuh"
#include "sgd_tail.cuh"

namespace ddrl {

// ---- weights: global flat (checkpoint order) -> shared (concatenated / transposed) --------------
__device__ void load_weights_flat(float* sm, const FcSmem& L, const float* __restrict__ th, int D, int A) {
    const FcOffsets o = fc_offsets(D, A);
    const int tid = threadIdx.x;
    for (int i = tid; i < L.x; i += NT) sm[i] = 0.f;   // pads (W1c rows D..Dp, WhT) must be zero
    __syncthreads();
    for (int j = tid; j < o.NP; j += NT) {
        const float w = th[j];
        int p0, p1;
        fc_img_pos(L, o, D, A, j, p0, p1);
        sm[p0] = w;
        if (p1 >= 0) sm[p1] = w;
    }
}

// ---- cp.async (LDGSTS): global -> shared without staging registers; completion via commit/wait groups ----------
__device__ __forceinline__ void cp_async4(float* smem_dst, const float* gsrc) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(d), "l"(gsrc));
}
__device__ __forceinline__ void cp_async16(float* smem_dst, const float* gsrc) {
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(d), "l"(gsrc));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;\n" ::: "memory"); }

__device__ __forceinline__ void load_weights_img(float* sm, const FcSmem& L, const float* __restrict__ img) {
    const int n4 = L.x >> 2;
    for (int i = threadIdx.x; i < n4; i += NT) cp_async16(sm + 4 * i, img + 4 * i);
}

// asynchronous x tile (no filter): rows row0.. -> xbuf[r*Dp + d]
__device__ __forceinline__ void prefetch_x_tile(float* xbuf, const float* __restrict__ obs, int64_t row0, int nrows, int D) {
    const int Dp = (D + 3) & ~3;
    const int n = nrows * D;
    const float* src = obs + row0 * D;
    for (int i = threadIdx.x; i < n; i += NT) {
        const int r = i / D, d = i - r * D;
        cp_async4(xbuf + r * Dp + d, src + i);
    }
}

// ---- register-tile micro kernels -------------------------------------------------------------
// acc[i][0..3] += sum_k A[i*lda + k] * B0[k*ldb + 0..3],  acc[i][4..7] likewise with B1;  K % 4 == 0.
__device__ __forceinline__ void mm_nn(const float* __restrict__ A, int lda, const float* __restrict__ B0,
                                      const float* __restrict__ B1, int ldb, int K, float (&acc)[4][8]) {
#pragma unroll 2
    for (int k = 0; k < K; k += 4) {
        float4 a[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) a[i] = *reinterpret_cast<const float4*>(A + i * lda + k);
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
            const float4 b0 = *reinterpret_cast<const float4*>(B0 + (k + kk) * ldb);
            const float4 b1 = *reinterpret_cast<const float4*>(B1 + (k + kk) * ldb);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const float av = kk == 0 ? a[i].x : kk == 1 ? a[i].y : kk == 2 ? a[i].z : a[i].w;
                acc[i][0] = fmaf(av, b0.x, acc[i][0]);
                acc[i][1] = fmaf(av, b0.y, acc[i][1]);
                acc[i][2] = fmaf(av, b0.z, acc[i][2]);
                acc[i][3] = fmaf(av, b0.w, acc[i][3]);
                acc[i][4] = fmaf(av, b1.x, acc[i][4]);
                acc[i][5] = fmaf(av, b1.y, acc[i][5]);
                acc[i][6] = fmaf(av, b1.z, acc[i][6]);
                acc[i][7] = fmaf(av, b1.w, acc[i][7]);
            }
        }
    }
}

// acc[i][j] += sum_r A[r*lda + i] * B{0,1}[r*ldb + j],  r = r0, r0+rs, ... < r1   (weight gradients).
__device__ __forceinline__ void mm_tn(const float* __restrict__ A, int lda, const float* __restrict__ B0,
                                      const float* __restrict__ B1, int ldb, int r0, int r1, int rs,
                                      float (&acc)[4][8]) {
#pragma unroll 4
    for (int r = r0; r < r1; r += rs) {
        const float4 a = *reinterpret_cast<const float4*>(A + r * lda);
        const float4 b0 = *reinterpret_cast<const float4*>(B0 + r * ldb);
        const float4 b1 = *reinterpret_cast<const float4*>(B1 + r * ldb);
        const float av[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            acc[i][0] = fmaf(av[i], b0.x, acc[i][0]);
            acc[i][1] = fmaf(av[i], b0.y, acc[i][1]);
            acc[i][2] = fmaf(av[i], b0.z, acc[i][2]);
            acc[i][3] = fmaf(av[i], b0.w, acc[i][3]);
            acc[i][4] = fmaf(av[i], b1.x, acc[i][4]);
            acc[i][5] = fmaf(av[i], b1.y, acc[i][5]);
            acc[i][6] = fmaf(av[i], b1.z, acc[i][6]);
            acc[i][7] = fmaf(av[i], b1.w, acc[i][7]);
        }
    }
}

__device__ __forceinline__ void zero_acc(float (&acc)[4][8]) {
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
}

// bias + tanh epilogue of a 4x8 tile, stored row-major into dst (stride LDH) at columns c0.. and c1..
__device__ __forceinline__ void tanh_store(float* sm_dst, const float* bias, int row0, int c0, int c1,
                                           const float (&acc)[4][8]) {
    const float4 b0 = *reinterpret_cast<const float4*>(bias + c0);
    const float4 b1 = *reinterpret_cast<const float4*>(bias + c1);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        float4 o0, o1;
        o0.x = tanhf(acc[i][0] + b0.x); o0.y = tanhf(acc[i][1] + b0.y);
        o0.z = tanhf(acc[i][2] + b0.z); o0.w = tanhf(acc[i][3] + b0.w);
        o1.x = tanhf(acc[i][4] + b1.x); o1.y = tanhf(acc[i][5] + b1.y);
        o1.z = tanhf(acc[i][6] + b1.z); o1.w = tanhf(acc[i][7] + b1.w);
        float* dst = sm_dst + (row0 + i) * LDH;
        *reinterpret_cast<float4*>(dst + c0) = o0;
        *reinterpret_cast<float4*>(dst + c1) = o1;
    }
}

// ---- forward of one tile: x (smem) -> h1, h2 (smem) -> out[r][0..2A] = logits, out[r][2A] = value --
__device__ __forceinline__ void forward_tile(float* sm, const FcSmem& L, int D, int A, int nrows) {
    const int Dp = (D + 3) & ~3;
    const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
    const int br = (tx >> 3) * H, c0 = br + (tx & 7) * 4, c1 = c0 + 32;
    const bool live = ty * 4 < nrows;  // rows of this thread hold data (8-row granularity per warp)
    float acc[4][8];
    if (live) {
        zero_acc(acc);
        mm_nn(sm + L.x + ty * 4 * Dp, Dp, sm + L.W1c + c0, sm + L.W1c + c1, HC, Dp, acc);
        tanh_store(sm + L.h1, sm + L.b1c, ty * 4, c0, c1, acc);
    }
    __syncthreads();
    if (live) {
        zero_acc(acc);
        mm_nn(sm + L.h1 + ty * 4 * LDH + br, LDH, sm + L.W2c + c0, sm + L.W2c + c1, HC, H, acc);
        tanh_store(sm + L.h2, sm + L.b2c, ty * 4, c0, c1, acc);
    }
    __syncthreads();
    // heads: item = (row r, output o); o == 2A is the value head reading the value branch of h2.
    const int A2 = 2 * A;
    for (int item = tid; item < TM * (A2 + 1); item += NT) {
        const int r = item & (TM - 1), o = item >> 6;
        if (r >= nrows) continue;
        const bool isv = o == A2;
        const float* hrow = sm + L.h2 + r * LDH + (isv ? H : 0);
        const float* w = isv ? sm + L.Wvo : sm + L.Wo + o;
        const int ws = isv ? 1 : A2;
        float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll 4
        for (int k = 0; k < H; k += 4) {
            const float4 hv = *reinterpret_cast<const float4*>(hrow + k);
            s0 = fmaf(hv.x, w[(k + 0) * ws], s0);
            s1 = fmaf(hv.y, w[(k + 1) * ws], s1);
            s2 = fmaf(hv.z, w[(k + 2) * ws], s2);
            s3 = fmaf(hv.w, w[(k + 3) * ws], s3);
        }
        sm[L.out + r * LDD + o] = ((s0 + s1) + (s2 + s3)) + (isv ? sm[L.bvo] : sm[L.bo + o]);
    }
    __syncthreads();
}

// ---- x tile: global -> shared, optional MeanStdFilter normalisation ---------------------------------
__device__ __forceinline__ void load_x_tile(float* sm, const FcSmem& L, const float* __restrict__ obs,
                                            float* __restrict__ obs_out, const double* snorm, float clip,
                                            int64_t row0, int nrows, int D) {
    const int Dp = (D + 3) & ~3;
    const int n = nrows * D;
    const float* src = obs + row0 * D;
    for (int i = threadIdx.x; i < n; i += NT) {
        const int r = i / D, d = i - r * D;
        float v = src[i];
        if (snorm) {
            v = (float)(((double)v - snorm[d]) * snorm[((D + 1) & ~1) + d]);
            if (clip > 0.f) v = fminf(fmaxf(v, -clip), clip);
        }
        if (obs_out) obs_out[row0 * D + i] = v;
        sm[L.x + r * Dp + d] = v;
    }
}

// =================================================================================================
// K1: grouped forward (+filter-normalise prologue, +DiagGaussian sample/logp epilogue)
// CUP = true (ddrl_fcnet_forward_coupled): the leg-coupled policy of SharedDecentralLegID — row r's mean logits are
// multiplied by coupling[node_id[r]] (one rounding, as leg_coupling_kernel) before they are stored and sampled from; an id
// outside 0..3 sets DDRL_STATUS_BAD_NODE and is coupled as id & 3.  The three trailing parameters are unused by <false>.
// =================================================================================================
template <bool CUP>
__global__ void __launch_bounds__(NT, 1)
fcnet_forward_kernel(const float* __restrict__ theta, const float* __restrict__ img, const float* __restrict__ obs,
                     const double* __restrict__ norm, float clip, int64_t R, int D, int A, float* __restrict__ obs_out,
                     float* __restrict__ logits, float* __restrict__ value, const float* __restrict__ eps,
                     float* __restrict__ action, float* __restrict__ logp, const int32_t* __restrict__ node_id,
                     const float* __restrict__ coupling, int* __restrict__ status) {
    extern __shared__ __align__(16) float sm[];
    const int p = blockIdx.y;
    const FcSmem L = fc_smem(D, A, norm != nullptr);
    const FcOffsets o = fc_offsets(D, A);
    const int tid = threadIdx.x;
    const int A2 = 2 * A;
    if (img) load_weights_img(sm, L, img + (int64_t)p * L.x);
    else load_weights_flat(sm, L, theta + (int64_t)p * o.NP, D, A);
    for (int i = tid; i < TM * ((D + 3) & ~3); i += NT) sm[L.x + i] = 0.f;
    double* snorm = nullptr;
    if (norm) {
        snorm = reinterpret_cast<double*>(sm + L.norm);
        const int Dd = (D + 1) & ~1;
        for (int i = tid; i < D; i += NT) {
            snorm[i] = norm[(int64_t)p * 2 * D + i];
            snorm[Dd + i] = norm[(int64_t)p * 2 * D + D + i];
        }
    }
    __syncthreads();
    const float* obs_p = obs + (int64_t)p * R * D;
    float* obs_out_p = obs_out ? obs_out + (int64_t)p * R * D : nullptr;
    const int64_t ntiles = (R + TM - 1) / TM;
    for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const int64_t row0 = t * TM;
        const int nrows = (int)min((int64_t)TM, R - row0);
        load_x_tile(sm, L, obs_p, obs_out_p, snorm, clip, row0, nrows, D);
        __syncthreads();
        forward_tile(sm, L, D, A, nrows);
        // epilogue ---------------------------------------------------------------------------------
        if (CUP && tid < nrows) {      // LegCoupling of row tid (this thread samples it below: no barrier in between)
            int nd = node_id[(int64_t)p * R + row0 + tid];
            if ((unsigned)nd > 3u) { atomicOr(status, DDRL_STATUS_BAD_NODE); nd &= 3; }
            float* mrow = sm + L.out + tid * LDD;
            mrow[0] = __fmul_rn(mrow[0], __ldg(coupling + 2 * nd));      // (never contracted into the sample's FMA)
            mrow[1] = __fmul_rn(mrow[1], __ldg(coupling + 2 * nd + 1));
        }
        if (eps && tid < nrows) {
            const int r = tid;
            const int64_t gr = (int64_t)p * R + row0 + r;
            float sz2 = 0.f, sls = 0.f;
            for (int i = 0; i < A; ++i) {
                const float mu = sm[L.out + r * LDD + i], ls = sm[L.out + r * LDD + A + i];
                const float sd = expf(ls);
                const float a = mu + sd * eps[gr * A + i];
                const float z = (a - mu) / sd;
                sz2 = fmaf(z, z, sz2);
                sls += ls;
                sm[L.dl + r * LDD + i] = a;
            }
            logp[gr] = -0.5f * sz2 - 0.5f * kLog2Pi * (float)A - sls;
        }
        if (CUP || eps) __syncthreads();
        if (logits)
            for (int i = tid; i < nrows * A2; i += NT) {
                const int r = i / A2, c = i - r * A2;
                logits[((int64_t)p * R + row0) * A2 + i] = sm[L.out + r * LDD + c];
            }
        if (value && tid < nrows) value[(int64_t)p * R + row0 + tid] = sm[L.out + tid * LDD + A2];
        if (eps)
            for (int i = tid; i < nrows * A; i += NT) {
                const int r = i / A, c = i - r * A;
                action[((int64_t)p * R + row0) * A + i] = sm[L.dl + r * LDD + c];
            }
        __syncthreads();
    }
}

// =================================================================================================
// K2/K6: fused forward + PPO loss + backward for one minibatch (all policies), per-CTA partial grads
// =================================================================================================
struct TrainArgs {
    const float *theta, *img, *obs, *actions, *old_logits, *old_logp, *vf_preds, *adv, *vtarg, *ext_dlogits, *ext_dvalue;
    int64_t R;
    int D, A, MB;
    const int32_t* mb_perm;
    int64_t perm_stride;
    const int32_t* step_ctr;
    const float* kl_coeff;
    ddrl_ppo_hyper hp;
    float* grad_part;
    double* stat_part;
    SgdTail tail;
};

// CUP = true: the leg-coupled policy of SharedDecentralLegID (see fcnet_train_tc2_cup_kernel, tc2.cu): the mean logits are
// scaled by c[node_id[r]] before the loss, the loss gradient of the mean logits by the same factor before the backward, and
// the table gradient sum_r dlogits[r][i] * pre[r][i] (per node) goes to flat indices [NP, NP + 8) of the partial.
// node_id [P][R]; the table is read from a.theta [P][NP + 8] (the weights themselves come from the image); an id outside
// 0..3 sets bit 128 of *a.tail.status.
__global__ void __launch_bounds__(NT, 1) fcnet_train_kernel(const TrainArgs a) {
    constexpr bool CUP = false;
    const int32_t* const node_id = nullptr;
#include "fcnet_train_body.inc"
}

__global__ void __launch_bounds__(NT, 1) fcnet_train_cup_kernel(const TrainArgs a, const int32_t* __restrict__ node_id) {
    constexpr bool CUP = true;
#include "fcnet_train_body.inc"
}

// flat theta -> packed shared-memory image (one thread per parameter)
__global__ void fcnet_pack_kernel(const float* __restrict__ theta, int D, int A, float* __restrict__ img) {
    const int p = blockIdx.y;
    const FcSmem L = fc_smem(D, A, false);
    const FcOffsets o = fc_offsets(D, A);
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= o.NP) return;
    int p0, p1;
    fc_img_pos(L, o, D, A, j, p0, p1);
    const float w = theta[(int64_t)p * o.NP + j];
    float* im = img + (int64_t)p * L.x;
    im[p0] = w;
    if (p1 >= 0) im[p1] = w;
}

}  // namespace ddrl

using namespace ddrl;

static int g_num_sms = 0;
static int num_sms() {
    if (g_num_sms == 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess) return 148;
        if (cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) g_num_sms = 148;
    }
    return g_num_sms;
}

extern "C" int ddrl_fcnet_num_params(int D, int A) {
    if (D < 1 || D > DDRL_MAX_OBS || A < 1 || A > DDRL_MAX_ACT) return DDRL_E_UNSUPPORTED_SHAPE;
    return fc_offsets(D, A).NP;
}

extern "C" int ddrl_fcnet_image_floats(int D, int A) {
    if (D < 1 || D > DDRL_MAX_OBS || A < 1 || A > DDRL_MAX_ACT) return DDRL_E_UNSUPPORTED_SHAPE;
    return fc_smem(D, A, false).x;
}

extern "C" int ddrl_fcnet_pack(const float* theta, int P, int D, int A, float* img, void* stream) {
    DDRL_REQUIRE(theta && img && P >= 1, DDRL_E_BADARG, "fcnet_pack: null pointer or bad P");
    DDRL_REQUIRE(D >= 1 && D <= DDRL_MAX_OBS && A >= 1 && A <= DDRL_MAX_ACT, DDRL_E_UNSUPPORTED_SHAPE,
                 "fcnet_pack: unsupported D=%d A=%d", D, A);
    const int NP = fc_offsets(D, A).NP;
    cudaMemsetAsync(img, 0, (size_t)P * fc_smem(D, A, false).x * sizeof(float), (cudaStream_t)stream);
    fcnet_pack_kernel<<<dim3((NP + 255) / 256, P), 256, 0, (cudaStream_t)stream>>>(theta, D, A, img);
    DDRL_CHECK_LAUNCH("fcnet_pack");
    return DDRL_OK;
}

// TrainArgs of the two FP32 train steps and their dynamic shared memory.
static int fp32_train_args(TrainArgs& a, size_t& smem, const char* who, const float* theta, const float* img, const float* obs,
                           const float* actions, const float* old_logits, const float* old_logp, const float* vf_preds,
                           const float* adv, const float* vtarg, const float* ext_dlogits, const float* ext_dvalue, int64_t R,
                           int D, int A, int MB, const int32_t* mb_perm, int64_t perm_stride, const int32_t* step_ctr,
                           const float* kl_coeff, const ddrl_ppo_hyper* hyper, float* grad_part, double* stat_part,
                           const ddrl_sgd_tail* tail) {
    a.theta = theta; a.img = img; a.obs = obs; a.actions = actions; a.old_logits = old_logits; a.old_logp = old_logp;
    a.vf_preds = vf_preds; a.adv = adv; a.vtarg = vtarg; a.ext_dlogits = ext_dlogits; a.ext_dvalue = ext_dvalue;
    a.R = R; a.D = D; a.A = A; a.MB = MB; a.mb_perm = mb_perm; a.perm_stride = perm_stride; a.step_ctr = step_ctr;
    a.kl_coeff = kl_coeff;
    a.hp = hyper ? *hyper : ddrl_ppo_hyper{0.f, 0.f, 0.f, 0.f, 1.f};
    a.grad_part = grad_part; a.stat_part = stat_part;
    a.tail = launch_tail(tail, false);
    smem = (size_t)fc_smem(D, A, false, true).total * sizeof(float);
    DDRL_REQUIRE(smem <= 227 * 1024, DDRL_E_UNSUPPORTED_SHAPE, "%s: shared memory %zu > 227 KB", who, smem);
    return DDRL_OK;
}

extern "C" int ddrl_ppo_train_step_coupled(const float* theta, const float* img, const int32_t* node_id, const float* obs,
                                           const float* actions, const float* old_logits, const float* old_logp,
                                           const float* vf_preds, const float* adv, const float* vtarg, int P, int64_t R,
                                           int D, int A, int MB, const int32_t* mb_perm, int64_t perm_stride,
                                           const int32_t* step_ctr, const float* kl_coeff, const ddrl_ppo_hyper* hyper,
                                           int ctas_per_policy, float* grad_part, double* stat_part, const ddrl_sgd_tail* tail,
                                           void* stream) {
    DDRL_REQUIRE(theta && img && node_id && obs && actions && old_logits && old_logp && vf_preds && adv && vtarg && kl_coeff &&
                     hyper && grad_part && P >= 1 && R >= 1 && MB >= 1 && ctas_per_policy >= 1,
                 DDRL_E_BADARG, "ppo_train_step_coupled: null pointer or bad P/R/MB/ctas");
    DDRL_REQUIRE(A == 2, DDRL_E_BADARG, "ppo_train_step_coupled: LegCoupling needs A = 2 (num_outputs == 4), got A=%d", A);
    DDRL_REQUIRE(P == 1, DDRL_E_BADARG, "ppo_train_step_coupled: the coupled model is one shared policy (P = 1), got P=%d", P);
    DDRL_REQUIRE(D >= 1 && D <= DDRL_MAX_OBS, DDRL_E_UNSUPPORTED_SHAPE, "ppo_train_step_coupled: unsupported D=%d", D);
    DDRL_REQUIRE(tail != nullptr, DDRL_E_BADARG, "ppo_train_step_coupled: the fused tail is required (NP + 8 parameters)");
    DDRL_REQUIRE(tail->theta == theta, DDRL_E_BADARG, "ppo_train_step_coupled: tail->theta must be theta");
    DDRL_REQUIRE(tail->status != nullptr, DDRL_E_BADARG,
                 "ppo_train_step_coupled: tail->status is required (it receives DDRL_STATUS_BAD_NODE for a node id outside 0..3)");
    const int rc = sgd_tail_check(tail, ctas_per_policy * P, "ppo_train_step_coupled");
    if (rc != DDRL_OK) return rc;
    DDRL_REQUIRE(tail->nsteps <= 1, DDRL_E_UNSUPPORTED_SHAPE, "ppo_train_step_coupled: nsteps > 1 is not supported by the FP32 kernel");
    DDRL_REQUIRE(!tail->ll_ws, DDRL_E_BADARG, "ppo_train_step_coupled: the LL tail is not supported with leg coupling");
    TrainArgs a;
    size_t smem = 0;
    if (int rc2 = fp32_train_args(a, smem, "ppo_train_step_coupled", theta, img, obs, actions, old_logits, old_logp, vf_preds, adv,
                                  vtarg, nullptr, nullptr, R, D, A, MB, mb_perm, perm_stride, step_ctr, kl_coeff, hyper,
                                  grad_part, stat_part, tail))
        return rc2;
    if (int rc2 = raise_smem_once<fcnet_train_cup_kernel>("ppo_train_step_coupled")) return rc2;
    fcnet_train_cup_kernel<<<dim3(ctas_per_policy, P), NT, smem, (cudaStream_t)stream>>>(a, node_id);
    DDRL_CHECK_LAUNCH("ppo_train_step_coupled");
    return DDRL_OK;
}

// The launch both FP32 forwards share (CUP = true: ddrl_fcnet_forward_coupled, P = 1).
template <bool CUP>
static int fcnet_forward_launch(const char* who, const float* theta, const float* img, const float* obs, const double* norm,
                                float clip, int P, int64_t R, int D, int A, float* obs_out, float* logits, float* value,
                                const float* eps, float* action, float* logp, const int32_t* node_id, const float* coupling,
                                int* status, void* stream) {
    if (R == 0) return DDRL_OK;
    const FcSmem L = fc_smem(D, A, norm != nullptr);
    const size_t smem = (size_t)L.total * sizeof(float);
    DDRL_REQUIRE(smem <= 227 * 1024, DDRL_E_UNSUPPORTED_SHAPE, "%s: shared memory %zu > 227 KB", who, smem);
    if (int rc = raise_smem_once<fcnet_forward_kernel<CUP>>(who)) return rc;
    const int64_t ntiles = (R + TM - 1) / TM;
    const int per_policy = (int)std::min<int64_t>(ntiles, std::max(1, num_sms() / P));
    fcnet_forward_kernel<CUP><<<dim3(per_policy, P), NT, smem, (cudaStream_t)stream>>>(
        theta, img, obs, norm, clip, R, D, A, obs_out, logits, value, eps, action, logp, node_id, coupling, status);
    DDRL_CHECK_LAUNCH(who);
    return DDRL_OK;
}

extern "C" int ddrl_fcnet_forward(const float* theta, const float* img, const float* obs, const double* norm,
                                  float clip, int P, int64_t R, int D, int A, float* obs_out, float* logits,
                                  float* value, const float* eps, float* action, float* logp, void* stream) {
    DDRL_REQUIRE((theta || img) && obs && P >= 1 && R >= 0, DDRL_E_BADARG, "fcnet_forward: null theta/obs or bad P/R");
    DDRL_REQUIRE(D >= 1 && D <= DDRL_MAX_OBS && A >= 1 && A <= DDRL_MAX_ACT, DDRL_E_UNSUPPORTED_SHAPE,
                 "fcnet_forward: unsupported D=%d A=%d (D<=%d, A<=%d, hiddens [64,64], tanh)", D, A, DDRL_MAX_OBS,
                 DDRL_MAX_ACT);
    DDRL_REQUIRE(!eps || (action && logp), DDRL_E_BADARG, "fcnet_forward: eps given without action/logp outputs");
    return fcnet_forward_launch<false>("fcnet_forward", theta, img, obs, norm, clip, P, R, D, A, obs_out, logits, value, eps,
                                       action, logp, nullptr, nullptr, nullptr, stream);
}

extern "C" int ddrl_fcnet_forward_coupled(const float* theta, const float* img, const int32_t* node_id, const float* coupling,
                                          const float* obs, const double* norm, float clip, int P, int64_t R, int D, int A,
                                          float* obs_out, float* logits, float* value, const float* eps, float* action,
                                          float* logp, int* status, void* stream) {
    DDRL_REQUIRE((theta || img) && node_id && coupling && obs && status && R >= 0, DDRL_E_BADARG,
                 "fcnet_forward_coupled: null theta/node_id/coupling/obs/status or bad R");
    DDRL_REQUIRE(A == 2, DDRL_E_BADARG, "fcnet_forward_coupled: LegCoupling needs A = 2 (num_outputs == 4), got A=%d", A);
    DDRL_REQUIRE(P == 1, DDRL_E_BADARG, "fcnet_forward_coupled: the coupled model is one shared policy (P = 1), got P=%d", P);
    DDRL_REQUIRE(D >= 1 && D <= DDRL_MAX_OBS, DDRL_E_UNSUPPORTED_SHAPE, "fcnet_forward_coupled: unsupported D=%d", D);
    DDRL_REQUIRE(!eps || (action && logp), DDRL_E_BADARG, "fcnet_forward_coupled: eps given without action/logp outputs");
    return fcnet_forward_launch<true>("fcnet_forward_coupled", theta, img, obs, norm, clip, P, R, D, A, obs_out, logits, value,
                                      eps, action, logp, node_id, coupling, status, stream);
}

extern "C" int ddrl_ppo_train_step(const float* theta, const float* img, const float* obs, const float* actions,
                                   const float* old_logits, const float* old_logp, const float* vf_preds,
                                   const float* adv, const float* vtarg, const float* ext_dlogits,
                                   const float* ext_dvalue, int P, int64_t R, int D, int A, int MB,
                                   const int32_t* mb_perm, int64_t perm_stride, const int32_t* step_ctr,
                                   const float* kl_coeff, const ddrl_ppo_hyper* hyper, int ctas_per_policy,
                                   float* grad_part, double* stat_part, const ddrl_sgd_tail* tail, void* stream) {
    DDRL_REQUIRE((theta || img) && obs && grad_part && P >= 1 && R >= 1 && MB >= 1 && ctas_per_policy >= 1,
                 DDRL_E_BADARG, "ppo_train_step: null pointer or bad P/R/MB/ctas");
    DDRL_REQUIRE(D >= 1 && D <= DDRL_MAX_OBS && A >= 1 && A <= DDRL_MAX_ACT, DDRL_E_UNSUPPORTED_SHAPE,
                 "ppo_train_step: unsupported D=%d A=%d", D, A);
    const bool ext = ext_dlogits != nullptr;
    DDRL_REQUIRE(ext ? (ext_dvalue != nullptr)
                     : (actions && old_logits && old_logp && vf_preds && adv && vtarg && kl_coeff && hyper),
                 DDRL_E_BADARG, "ppo_train_step: missing batch arrays for the %s path", ext ? "external-gradient" : "PPO");
    if (tail) {
        DDRL_REQUIRE(!ext, DDRL_E_BADARG, "ppo_train_step: the fused tail cannot be combined with external gradients");
        const int rc = sgd_tail_check(tail, ctas_per_policy * P, "ppo_train_step");
        if (rc != DDRL_OK) return rc;
        DDRL_REQUIRE(tail->nsteps <= 1, DDRL_E_UNSUPPORTED_SHAPE, "ppo_train_step: nsteps > 1 is not supported by the FP32 kernel");
    }
    TrainArgs a;
    size_t smem = 0;
    if (int rc = fp32_train_args(a, smem, "ppo_train_step", theta, img, obs, actions, old_logits, old_logp, vf_preds, adv, vtarg,
                                 ext_dlogits, ext_dvalue, R, D, A, MB, mb_perm, perm_stride, step_ctr, kl_coeff, hyper,
                                 grad_part, stat_part, tail))
        return rc;
    if (int rc = raise_smem_once<fcnet_train_kernel>("ppo_train_step")) return rc;
    fcnet_train_kernel<<<dim3(ctas_per_policy, P), NT, smem, (cudaStream_t)stream>>>(a);
    DDRL_CHECK_LAUNCH("ppo_train_step");
    return DDRL_OK;
}

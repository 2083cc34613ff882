// Tensor-core FCNet step, "ping-pong" schedule (sm_100a, tcgen05 + TMEM): the PPO training step of all policies as ONE
// persistent kernel, and (template flag FWD) the inference forward.
//
// Same operand layouts, scales and arithmetic as fcnet_train_tc_kernel (tc.cu) — fused forward + PPO loss + backward,
// per-CTA partial gradients in flat checkpoint order — but BOTH branches of the network (policy MLP and value MLP) are
// resident at once and software-pipelined against each other:
//
//     issue F1(pol), F1(val) | wait pol -> tanh epilogue(pol) -> issue F2(pol) | wait val -> tanh epilogue(val) -> issue F2(val) | ...
//
//   * 16 epilogue warps (TMEM -> tanh / (1-h^2) -> fp16 hi/lo -> shared memory) + 4 MMA-issue warps.  While the epilogue
//     warps work on one branch the tensor core executes the other branch's GEMMs; each branch has its own accumulator
//     columns and its own mbarrier (expected arrivals = the 4 issuers).  The issuers are warps of their own because a lane
//     that shares a warp with lanes spinning in mbarrier.try_wait gets its issue delayed by 0.5-2 us, and there are four of
//     them because one thread issues a tcgen05.mma only every ~72 cycles whatever its shape (tests/umma_bench.py).
//   * the two PPO-loss halves (policy part on warps 0-3, value part on warps 4-7) run concurrently.
//   * H1/H2 of both branches live in shared memory (128 KB); DL, the observation staging and (A = 8) the old logits reuse
//     space that is dead at the time (fcnet_tc_layout.cuh): D <= 47, every published architecture (tc2_eligible).
//   * the weight-gradient GEMMs stack the hi | lo halves of their A operand along M (tc_gemm_stack_u: one M = 128 MMA gives
//     A_hi^T B and A_lo^T B; dependent chains of 16 / 8 instead of 24 / 16 MMAs), and the four MMA-issue warps — idle between
//     two hand-offs — read the finished accumulators out of TMEM and stage the partial gradient in shared memory in the gaps
//     of their issue schedule; the epilogue warps copy it out (two staging halves added on the way) while the last MMAs run.
//   * the launch runs a.tail.nsteps consecutive optimizer steps: per step the fused tail (sgd_tail.cuh) reduces the
//     partial gradients over the CTAs of a policy (by default they are ADDED into one vector per policy at L2 by the
//     copy-out, ddrl_sgd_tail.grad_acc), all-reduces them over NVLink peer memory (world > 1), clips and applies Adam; the
//     CTAs of a policy meet at a barrier before they reload the updated weight image.  The next step's inputs are requested
//     behind the tail.
//   * the step is sensitive to CODE SIZE (every warp walks ~4 000 instructions once per ~23 us step, far more than the
//     32 KB instruction cache holds): issue loops are not unrolled, debug stamps sit behind the DBG template flag.
//   * FWD = true: forward-only over all rows of each policy (filter normalise in the X split, DiagGaussian sample + logp in
//     place of the loss) — ddrl_fcnet_forward_tc.
#include <algorithm>

#include "tc_common.cuh"

namespace ddrl {

// TMEM columns: per-branch forward/backward accumulator, head outputs, and the weight-gradient accumulators
// GW1 and GWH exist twice per branch ([2b + s]: s = 0 takes the hi*hi product, s = 1 the two cross products) so that two
// MMA warps can issue one weight-gradient GEMM concurrently; the halves are added at the write-out.
constexpr int T2_DACC = 0, T2_HOUT = 128, T2_GW2 = 160, T2_GW1 = 288, T2_GB2 = 416, T2_GWH = 448, T2_TMEM_COLS = 512;
constexpr int T2_NMMA = 4;                   // MMA-issue warps: one thread issues a tcgen05.mma every ~72 cycles whatever its
                                             // shape (tests/umma_bench.py), so the ~270 MMAs of a tile are spread over 4 issuers
constexpr int T2_NT = TC_NT + 32 * T2_NMMA;  // 16 epilogue warps + the MMA-issue warps
constexpr int T2_MMA_WARP = TC_NT / 32;      // first MMA warp (16); these warps never touch an accumulator

// Epilogue math in packed FP32 pairs (sm_100a FFMA2 / FADD2 / FMUL2: one issue slot for two FP32 operations).
// tanh(x) = 1 - 2 r, r = 1 / (2^(2 log2(e) x) + 1): MUFU ex2 + rcp, absolute error <= 2.4e-7 over the whole range (tanhf:
// 1.2e-7; 2^y overflows to +inf -> r = 0 -> 1, underflows to 0 -> r = 1 -> -1, so no |x| / copysign is needed).  The
// cancellation near 0 costs RELATIVE accuracy only, and the activations are cut to ~22 bits (fp16 hi + lo, 2.4e-7 absolute)
// right afterwards, so the odd-polynomial branch of tanhf buys nothing here.
constexpr float kT2TanhIn = 2.885390081777927f;      // 2 log2(e)
__device__ __forceinline__ float2 t2_tanh2(float2 y) {      // y = 2 log2(e) x
    float2 t, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(t.x) : "f"(y.x));
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(t.y) : "f"(y.y));
    t = __fadd2_rn(t, make_float2(1.f, 1.f));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r.x) : "f"(t.x));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r.y) : "f"(t.y));
    return __ffma2_rn(make_float2(-2.f, -2.f), r, make_float2(1.f, 1.f));
}
// (x0, x1) (already scaled, inside the fp16 range) -> fp16 hi pair / lo pair
__device__ __forceinline__ void t2_split2v(float2 x, uint32_t& h, uint32_t& l) {
    const __half2 hh = __floats2half2_rn(x.x, x.y);
    const float2 hf = __half22float2(hh);
    const float2 d = __fadd2_rn(x, make_float2(-hf.x, -hf.y));
    const __half2 ll = __floats2half2_rn(d.x, d.y);
    h = *reinterpret_cast<const uint32_t*>(&hh);
    l = *reinterpret_cast<const uint32_t*>(&ll);
}

// Forward epilogue of this thread's 16 columns: act = tanh(acc * inv_in + bias) -> fp16 hi/lo (x TC_SH), chunked [128][64].
__device__ __noinline__ void t2_epi_tanh(uint32_t taddr, const float* bias, float inv_in, unsigned char* dhi, unsigned char* dlo,
                                         int row, int cq) {
    const float2 k2 = make_float2(inv_in * kT2TanhIn, inv_in * kT2TanhIn), c2 = make_float2(kT2TanhIn, kT2TanhIn),
                 sh = make_float2(TC_SH, TC_SH);
    // (two x8 TMEM loads, not one x16: measured 0.55 us per step FASTER — the second half's load overlaps the first half's math)
#pragma unroll 1
    for (int c = 0; c < 2; ++c) {
        float v[8];
        umma::tmem_ld8(taddr + 8 * c, v);
        const float4 b0 = *reinterpret_cast<const float4*>(bias + 8 * c);
        const float4 b1 = *reinterpret_cast<const float4*>(bias + 8 * c + 4);
        const float2 bb[4] = {make_float2(b0.x, b0.y), make_float2(b0.z, b0.w), make_float2(b1.x, b1.y), make_float2(b1.z, b1.w)};
        uint32_t h[4], l[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float2 y = __ffma2_rn(make_float2(v[2 * j], v[2 * j + 1]), k2, __fmul2_rn(bb[j], c2));
            t2_split2v(__fmul2_rn(t2_tanh2(y), sh), h[j], l[j]);          // |tanh| <= 1: always inside the fp16 range
        }
        const int off = ((2 * cq + c) * TC_ROWS + row) * 16;
        *reinterpret_cast<uint4*>(dhi + off) = make_uint4(h[0], h[1], h[2], h[3]);
        *reinterpret_cast<uint4*>(dlo + off) = make_uint4(l[0], l[1], l[2], l[3]);
    }
}

// Backward epilogue: g = acc * inv_in * (1 - h^2), h re-read from the buffer it then overwrites (fp16 hi/lo x out_scale).
// Returns true if |g * out_scale| left the fp16 range.
__device__ __noinline__ bool t2_epi_grad(uint32_t taddr, float inv_in, float out_scale, unsigned char* bhi, unsigned char* blo,
                                         int row, int cq) {
    float mx = 0.f;
    const float2 ki = make_float2(inv_in, inv_in), ks = make_float2(1.f / TC_SH, 1.f / TC_SH), os = make_float2(out_scale, out_scale),
                 one = make_float2(1.f, 1.f);
#pragma unroll 1
    for (int c = 0; c < 2; ++c) {
        float v[8];
        umma::tmem_ld8(taddr + 8 * c, v);
        const int off = ((2 * cq + c) * TC_ROWS + row) * 16;
        const uint4 qh = *reinterpret_cast<const uint4*>(bhi + off), ql = *reinterpret_cast<const uint4*>(blo + off);
        const __half2* hp = reinterpret_cast<const __half2*>(&qh);
        const __half2* lp = reinterpret_cast<const __half2*>(&ql);
        uint32_t h[4], l[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const float2 act = __fmul2_rn(__fadd2_rn(__half22float2(hp[j]), __half22float2(lp[j])), ks);
            const float2 om = __ffma2_rn(make_float2(-act.x, -act.y), act, one);                    // 1 - h^2
            const float2 g = __fmul2_rn(__fmul2_rn(make_float2(v[2 * j], v[2 * j + 1]), ki), om);
            mx = fmaxf(mx, fmaxf(fabsf(g.x), fabsf(g.y)));
            t2_split2v(__fmul2_rn(g, os), h[j], l[j]);      // an overflow of the fp16 range is reported through the return value
        }
        *reinterpret_cast<uint4*>(bhi + off) = make_uint4(h[0], h[1], h[2], h[3]);
        *reinterpret_cast<uint4*>(blo + off) = make_uint4(l[0], l[1], l[2], l[3]);
    }
    return !(mx * out_scale <= 60000.f);
}

// Shared-memory stores through an explicit shared::cta address.  The staging base is passed through an empty asm statement
// ("laundered") so that ptxas keeps it in ONE register: left visible, the base is re-derived from D at every store of the
// write-out (the kernel sits at its 96-register cap) — ~20 integer instructions per stored element, which made the
// write-out issue bound (1.5 us for two TMEM loads and 16 stores per thread).
__device__ __forceinline__ uint32_t t2_launder(uint32_t x) { asm volatile("" : "+r"(x)); return x; }
__device__ __forceinline__ void t2_sts(uint32_t a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); }
__device__ __forceinline__ void t2_sts4(uint32_t a, float x, float y, float z, float w) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(x), "f"(y), "f"(z), "f"(w) : "memory");
}
__device__ __forceinline__ float4 t2_lds4(uint32_t a) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a) : "memory");
    return v;
}

// (DBG is a template flag of the kernel: the ~50 stamp sites cost ~500 instructions, and the step is sensitive to its code size —
// the kernel is ~8 000 instructions executed once per step against a 32 KB instruction cache.  Only the bench shape has a DBG
// instantiation, tests/phase_clock.py.)
#define T2_STAMP(i)                                                                        \
    do {                                                                                   \
        if constexpr (DBG) {                                                               \
            if (a.dbg_clock && threadIdx.x == 0 && blockIdx.x == 0 && blockIdx.y == 0) a.dbg_clock[i] = clock64(); \
        }                                                                                  \
    } while (0)

// every CTA: globaltimer stamps (comparable across SMs) at a few points of the step -> dbg_clock[64 + 8 * cta + k]
__device__ __forceinline__ long long t2_gtime() {
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
#define T2_GSTAMP(k)                                                                                     \
    do {                                                                                                 \
        if constexpr (DBG) {                                                                             \
            if (a.dbg_clock && threadIdx.x == 0) a.dbg_clock[64 + 8 * (blockIdx.y * gridDim.x + blockIdx.x) + (k)] = t2_gtime(); \
        }                                                                                                \
    } while (0)

// FWD = true: forward-only (inference) mode — the same F1 / tanh / F2 / tanh / heads pipeline over ALL rows of each policy
// (a.MB = a.R), filter normalisation in the X split, DiagGaussian sample + logp in place of the loss, nothing after it.
// LL = true: the barrier-free "LL" tail (sgd_tail.cuh); its own instantiation so that the classic kernel keeps its register
// allocation (the kernel sits at the 96-register limit of 640 threads: the merged variant spilled and lost 3 us per step).
// DT > 0: the observation width as a compile-time constant (the launcher instantiates the ten (D, A) pairs of the published
// architectures, policies.ARCHITECTURES; DT = 0 reads a.D).  Every shared-memory offset, image offset and flat-parameter offset
// is a function of (D, A): with D in a register ptxas — at the kernel's 96-register cap — re-derived them from D at nearly
// every use (~20 integer instructions per staged element in the x split and the write-out); as constants they cost nothing.
// CUP = true: the leg-coupled policy of SharedDecentralLegID (models/coupling_net_glorot_uniform_init.py:11-30,135; A = 2,
// no clusters, no LL tail, fused tail required).  The mean logits are scaled by the trainable table c[node][i] before the
// loss, the loss gradient of the mean logits by the same factor before it enters the backward, and the table's own gradient
// sum_r dlogits[r][i] * pre[r][i] (per node) goes to flat indices [NP, NP + 8) of the partial: the step's parameter vector
// is [NP + 8] (FCNet variables, then leg_coupling [4][2]), and the fused tail clips and steps all of it.
//   node_id  [P][R] int32 in the batch's row order (rows of a tile are staged in shared memory with the loss inputs)
//   cup_theta  the flat parameter vector [P][NP + 8]: the table is read from it at the start of every step (after barrier C)
template <int A, bool FWD, bool LL, int DT, bool DBG>
__global__ void __launch_bounds__(T2_NT, 1) fcnet_train_tc2_kernel(const __grid_constant__ TcTrainArgs a) {
    constexpr bool CUP = false;
    const int32_t* const node_id = nullptr;
    const float* const cup_theta = nullptr;
    const float* const coupling = nullptr;
#include "tc2_step_body.inc"
}

// the leg-coupled step (SharedDecentralLegID): A = 2, D = DT
template <int DT>
__global__ void __launch_bounds__(T2_NT, 1) fcnet_train_tc2_cup_kernel(const __grid_constant__ TcTrainArgs a,
                                                                       const int32_t* __restrict__ node_id,
                                                                       const float* __restrict__ cup_theta) {
    constexpr int A = 2;
    constexpr bool FWD = false, LL = false, DBG = false, CUP = true;
    const float* const coupling = nullptr;
#include "tc2_step_body.inc"
}

// the leg-coupled inference forward (ddrl_fcnet_forward_tc_coupled): the FWD pipeline with the mean logits scaled by
// coupling[node_id[r]] before they are stored and sampled from.  node_id [R] (staged with the tile's noise), coupling [4][2].
// D is read from a.D, as in the uncoupled forward: with D as a compile-time constant (DT = 19, 20) ptxas spilled 16 bytes.
__global__ void __launch_bounds__(T2_NT, 1) fcnet_forward_tc2_cup_kernel(const __grid_constant__ TcTrainArgs a,
                                                                         const int32_t* __restrict__ node_id,
                                                                         const float* __restrict__ coupling) {
    constexpr int A = 2, DT = 0;
    constexpr bool FWD = true, LL = false, DBG = false, CUP = true;
    const float* const cup_theta = nullptr;
#include "tc2_step_body.inc"
}

static int g_tc2_cluster = 0;    // 0 = off (default: measured slower, DESIGN.md §4.1), -1 = automatic (largest of 16, 8, 4, 2 that
                                 // divides G and is co-resident), else the forced size

template <int A, bool FWD, bool LL, int DT = 0, bool DBG = false>
static int launch_tc2_t(const TcTrainArgs& a, int P, int G, size_t smem, cudaStream_t st, int* used_cluster) {
    constexpr auto kern = fcnet_train_tc2_kernel<A, FWD, LL, DT, DBG>;
    if (int rc = raise_smem_once<kern>("ppo_train_step_tc")) return rc;
    static bool cluster_attr = false;
    if (!cluster_attr) {
        cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);   // clusters of 16 (opt-in size)
        cudaGetLastError();
        cluster_attr = true;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(G, P);
    cfg.blockDim = dim3(T2_NT);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    // cluster size: cached per (P, G); the persistent / fused-tail kernel needs ALL clusters co-resident
    static int cache_P = -1, cache_G = -1, cache_cs = 1, cache_req = -2;
    if (cache_P != P || cache_G != G || cache_req != g_tc2_cluster) {
        int best = 1;
        const int cand[4] = {16, 8, 4, 2};
        for (int c = 0; c < 4; ++c) {
            const int csz = cand[c];
            if (g_tc2_cluster >= 0 && csz != g_tc2_cluster) continue;
            if (G % csz) continue;
            at[0].val.clusterDim.x = csz;
            int ncl = 0;
            if (cudaOccupancyMaxActiveClusters(&ncl, kern, &cfg) != cudaSuccess) { cudaGetLastError(); continue; }
            if (ncl * csz >= G * P) { best = csz; break; }
        }
        cache_P = P; cache_G = G; cache_cs = best; cache_req = g_tc2_cluster;
    }
    // without the fused tail the caller reduces G per-CTA partials itself (ddrl_grad_reduce): no cluster pre-reduction
    const int cs_use = (a.tail.theta && !LL) ? cache_cs : 1;
    at[0].val.clusterDim.x = cs_use;
    if (used_cluster) *used_cluster = cs_use;
    if (cudaLaunchKernelEx(&cfg, kern, a) != cudaSuccess) {
        set_error("ppo_train_step_tc: cluster launch (size %d) failed: %s", cs_use, cudaGetErrorString(cudaGetLastError()));
        return DDRL_E_CUDA;
    }
    return DDRL_OK;
}

static int g_tc2_last_cluster = 0;

bool tc2_clusters_requested() { return g_tc2_cluster != 0; }

int launch_tc2(const TcTrainArgs& a, int P, int G, cudaStream_t st) {
    const size_t smem = (size_t)tc2_smem(a.D, a.A).total;
    int* const used = &g_tc2_last_cluster;
    const char* const unsupported = "ppo_train_step_tc: ping-pong kernel supports A in {1,2,4,8}";
    // LL tail: fused tail with an LL workspace, no thread-block clusters requested, one slice element per thread
    if (a.tail.theta && a.tail.ll_ws && g_tc2_cluster == 0 && sgd_slice_len(fc_offsets(a.D, a.A).NP, G) <= T2_NT)
        return dispatch_A(a.A, unsupported,
                          [&](auto A_) { return launch_tc2_t<decltype(A_)::value, false, true>(a, P, G, smem, st, used); });
    // the published architectures (policies.ARCHITECTURES: obs width with / without the target velocity, action width)
    if (a.dbg_clock && a.D == 19 && a.A == 2) return launch_tc2_t<2, false, false, 19, true>(a, P, G, smem, st, used);
#define T2_PUBLISHED(DD, AA) \
    if (a.D == DD && a.A == AA) return launch_tc2_t<AA, false, false, DD>(a, P, G, smem, st, used);
    T2_PUBLISHED(19, 2) T2_PUBLISHED(20, 2) T2_PUBLISHED(27, 2) T2_PUBLISHED(28, 2) T2_PUBLISHED(35, 2) T2_PUBLISHED(36, 2)
    T2_PUBLISHED(27, 4) T2_PUBLISHED(28, 4) T2_PUBLISHED(43, 8) T2_PUBLISHED(44, 8)
#undef T2_PUBLISHED
    return dispatch_A(a.A, unsupported,
                      [&](auto A_) { return launch_tc2_t<decltype(A_)::value, false, false>(a, P, G, smem, st, used); });
}

// leg-coupled step: no clusters, no LL tail (the entry point rejects both); instantiated for SharedDecentralLegID's D = 19, 20
template <int DT>
static int launch_tc2_cup_t(const TcTrainArgs& a, const int32_t* node_id, const float* theta, int P, int G, cudaStream_t st) {
    if (int rc = raise_smem_once<fcnet_train_tc2_cup_kernel<DT>>("ppo_train_step_tc_coupled")) return rc;
    const size_t smem = (size_t)tc2_smem(DT, 2, true).total;
    fcnet_train_tc2_cup_kernel<DT><<<dim3(G, P), T2_NT, smem, st>>>(a, node_id, theta);
    g_tc2_last_cluster = 1;
    return DDRL_OK;
}

int launch_tc2_cup(const TcTrainArgs& a, const int32_t* node_id, const float* theta, int P, int G, cudaStream_t st) {
    if (g_tc2_cluster != 0) {
        set_error("ppo_train_step_tc_coupled: thread-block clusters are not supported with leg coupling (ddrl_tc_set_cluster(1))");
        return DDRL_E_BADARG;
    }
    if (a.A == 2 && a.D == 19) return launch_tc2_cup_t<19>(a, node_id, theta, P, G, st);
    if (a.A == 2 && a.D == 20) return launch_tc2_cup_t<20>(a, node_id, theta, P, G, st);
    set_error("ppo_train_step_tc_coupled: instantiated for A = 2 and D in {19, 20} (SharedDecentralLegID), got D=%d A=%d", a.D, a.A);
    return DDRL_E_UNSUPPORTED_SHAPE;
}

int launch_tc2_forward_cup(const TcTrainArgs& a, const int32_t* node_id, const float* coupling, int G, cudaStream_t st) {
    if (int rc = raise_smem_once<fcnet_forward_tc2_cup_kernel>("fcnet_forward_tc_coupled")) return rc;
    fcnet_forward_tc2_cup_kernel<<<dim3(G, 1), T2_NT, (size_t)tc2_smem(a.D, 2, true).total, st>>>(a, node_id, coupling);
    return DDRL_OK;
}

int launch_tc2_forward(const TcTrainArgs& a, int P, int G, cudaStream_t st) {
    const size_t smem = (size_t)tc2_smem(a.D, a.A).total;
    int dummy = 0;
    return dispatch_A(a.A, "fcnet_forward_tc: A must be 1, 2, 4 or 8",
                      [&](auto A_) { return launch_tc2_t<decltype(A_)::value, true, false>(a, P, G, smem, st, &dummy); });
}

}  // namespace ddrl

extern "C" int ddrl_tc_set_cluster(int cluster_size) {
    DDRL_REQUIRE(cluster_size == -1 || cluster_size == 1 || cluster_size == 2 || cluster_size == 4 || cluster_size == 8 ||
                     cluster_size == 16, DDRL_E_BADARG, "tc_set_cluster: size must be -1 (auto), 1, 2, 4, 8 or 16");
    ddrl::g_tc2_cluster = cluster_size == 1 ? 0 : cluster_size;
    return DDRL_OK;
}

extern "C" int ddrl_tc_last_cluster(void) { return ddrl::g_tc2_last_cluster; }

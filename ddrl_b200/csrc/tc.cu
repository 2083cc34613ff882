// tcgen05 tensor-core path (sm_100a): UMMA self test + (later) the tensor-core FCNet step.
#include <algorithm>

#include "common.cuh"
#include "umma.cuh"

namespace ddrl {

// D[128][N] = sum_k A(m,k) * B(n,k) on the 5th-gen tensor cores through TMEM, with the operands staged in the
// chunked shared-memory layout of umma.cuh.  A(m,k) = Abuf[m][k] (K-major) or Abuf[k][m] (MN-major view of the same
// kind of buffer); B alike.  split != 0: every operand is split into fp16 (hi, lo) and three products
// hi*hi + hi*lo + lo*hi are accumulated in FP32 (the precision scheme of the tensor-core training step).
__global__ void __launch_bounds__(128, 1)
umma_selftest_kernel(const float* __restrict__ A, int ra, int ca, const float* __restrict__ B, int rb, int cb, int M, int N,
                     int K, int a_mn, int b_mn, int split, float* __restrict__ D, int* __restrict__ status) {
    extern __shared__ __align__(128) unsigned char smraw[];
    __shared__ uint32_t tmem_slot;
    __shared__ __align__(8) uint64_t mbar;
    __half* sAh = reinterpret_cast<__half*>(smraw);
    __half* sAl = sAh + ra * ca;
    __half* sBh = sAl + ra * ca;
    __half* sBl = sBh + rb * cb;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    for (int i = tid; i < ra * ca; i += blockDim.x) {
        const int r = i / ca, c = i - r * ca;
        __half hi, lo;
        umma::split_f16(A[i], hi, lo);
        const int o = ((c >> 3) * ra + r) * 8 + (c & 7);
        sAh[o] = hi; sAl[o] = lo;
    }
    for (int i = tid; i < rb * cb; i += blockDim.x) {
        const int r = i / cb, c = i - r * cb;
        __half hi, lo;
        umma::split_f16(B[i], hi, lo);
        const int o = ((c >> 3) * rb + r) * 8 + (c & 7);
        sBh[o] = hi; sBl[o] = lo;
    }
    const uint32_t ncols = N <= 32 ? 32 : N <= 64 ? 64 : N <= 128 ? 128 : 256;
    if (warp == 0) umma::tmem_alloc(&tmem_slot, ncols);
    if (tid == 0) { umma::mbar_init(&mbar, 1); umma::fence_mbar_init(); }
    umma::fence_async_smem();
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t taddr = tmem_slot;
    if (tid == 0) {
        const uint32_t idesc = umma::idesc_f16(M, N, a_mn != 0, b_mn != 0);
        const int nprod = split ? 3 : 1;
        bool acc = false;
        for (int pr = 0; pr < nprod; ++pr) {
            const __half* pa = pr == 2 ? sAl : sAh;
            const __half* pb = pr == 1 ? sBl : sBh;
            for (int ks = 0; ks < K / 16; ++ks) {
                // K-major: 2 chunks of 8 per MMA, chunk stride rows*16 B.  MN-major: 16 K rows, 16 B each.
                const uint32_t aoff = a_mn ? ks * 16 * 16 : ks * 2 * ra * 16;
                const uint32_t boff = b_mn ? ks * 16 * 16 : ks * 2 * rb * 16;
                const uint64_t ad = a_mn ? umma::desc_mnmajor(umma::smem_u32(pa) + aoff, ra) : umma::desc_kmajor(umma::smem_u32(pa) + aoff, ra);
                const uint64_t bd = b_mn ? umma::desc_mnmajor(umma::smem_u32(pb) + boff, rb) : umma::desc_kmajor(umma::smem_u32(pb) + boff, rb);
                umma::mma_f16(taddr, ad, bd, idesc, acc);
                acc = true;
            }
        }
        umma::mma_commit(&mbar);
    }
    const bool ok = umma::mbar_wait(&mbar, 0);
    umma::fence_after_sync();
    if (!ok) {
        if (tid == 0) *status = 1;   // timed out: report, do not touch TMEM results
    } else {
        for (int c0 = 0; c0 < N; c0 += 32) {
            float v[32];
            umma::tmem_ld32(taddr + ((uint32_t)(warp * 32) << 16) + c0, v);
#pragma unroll
            for (int j = 0; j < 32; ++j)
                if (c0 + j < N) D[(warp * 32 + lane) * N + c0 + j] = v[j];
        }
        if (tid == 0) *status = 0;
    }
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 0) umma::tmem_dealloc(taddr, ncols);
}

}  // namespace ddrl

using namespace ddrl;

extern "C" int ddrl_umma_selftest(const float* A, int ra, int ca, const float* B, int rb, int cb, int M, int N, int K,
                                  int a_mn, int b_mn, int split, float* D, int* status, void* stream) {
    DDRL_REQUIRE(A && B && D && status, DDRL_E_BADARG, "umma_selftest: null pointer");
    DDRL_REQUIRE(ra % 8 == 0 && rb % 8 == 0 && ca % 8 == 0 && cb % 8 == 0 && K % 16 == 0 && N % 16 == 0 && N >= 16 && N <= 256,
                 DDRL_E_UNSUPPORTED_SHAPE, "umma_selftest: shapes must be multiples of 8 (rows/cols), 16 (K, N)");
    DDRL_REQUIRE(M == 64 || M == 128, DDRL_E_UNSUPPORTED_SHAPE, "umma_selftest: M must be 64 or 128");
    DDRL_REQUIRE((a_mn ? (ca >= M && ra >= K) : (ra >= M && ca >= K)) && (b_mn ? (cb >= N && rb >= K) : (rb >= N && cb >= K)),
                 DDRL_E_UNSUPPORTED_SHAPE, "umma_selftest: buffer shapes do not cover M x N x K");
    const size_t smem = (size_t)(ra * ca + rb * cb) * 2 * sizeof(__half) + 128;
    DDRL_REQUIRE(smem <= 200 * 1024, DDRL_E_UNSUPPORTED_SHAPE, "umma_selftest: %zu bytes of shared memory", smem);
    static bool attr = false;
    if (!attr) {
        if (cudaFuncSetAttribute(umma_selftest_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024) != cudaSuccess) {
            set_error("umma_selftest: cannot raise dynamic shared memory");
            return DDRL_E_CUDA;
        }
        attr = true;
    }
    umma_selftest_kernel<<<1, 128, smem, (cudaStream_t)stream>>>(A, ra, ca, B, rb, cb, M, N, K, a_mn, b_mn, split, D, status);
    DDRL_CHECK_LAUNCH("umma_selftest");
    return DDRL_OK;
}

// Micro-benchmark: `reps` back-to-back tcgen05.mma (kind::f16, M x N x 16) issued by one thread on garbage operands of the
// chunked layout; cycles[0] = issue loop only, cycles[1] = issue + commit + completion wait.  Sizes the MMA schedule.
namespace ddrl {
__global__ void __launch_bounds__(128, 1) umma_bench_kernel(int M, int N, int a_mn, int b_mn, int reps, int ksteps,
                                                            long long* __restrict__ cycles, int* __restrict__ status) {
    extern __shared__ __align__(128) unsigned char smraw[];
    __shared__ uint32_t tmem_slot;
    __shared__ __align__(8) uint64_t mbar;
    const int tid = threadIdx.x, warp = tid >> 5;
    for (int i = tid; i < 96 * 1024 / 4; i += blockDim.x) reinterpret_cast<uint32_t*>(smraw)[i] = 0x3c003c00u;   // 1.0h
    if (warp == 0) umma::tmem_alloc(&tmem_slot, 512);
    umma::fence_async_smem();
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t taddr = tmem_slot;
    long long t0 = 0, t1 = 0, t2 = 0;
    bool ok = true;
    // ksteps encodes the experiment: bits [0,8) k-steps per rep; bit 8: elect.sync instead of `lane == 0`;
    // bits [9,12): accumulators - 1 the issuing thread cycles through (independent MMA chains, N columns apart);
    // bits [12,14): log2(issuing warps) — warp w issues the same stream into its own accumulator set (128 columns apart)
    // bit 14: warp-uniform issue (umma::mma_f16_elect, operands made provably uniform with __shfl_sync)
    const int mode = (ksteps >> 8) & 1, nacc = ((ksteps >> 9) & 7) + 1, nwarps = 1 << ((ksteps >> 12) & 3);
    const bool uniform = (ksteps >> 14) & 1;
    ksteps &= 255;
    if (tid == 0) { umma::mbar_init(&mbar, nwarps); umma::fence_mbar_init(); }
    __syncthreads();
    if (warp < nwarps) {
        const uint32_t idesc = umma::idesc_f16(M, N, a_mn != 0, b_mn != 0);
        const uint32_t sa = umma::smem_u32(smraw), sb = sa + 48 * 1024;
        const uint64_t ad0 = a_mn ? umma::desc_mnmajor(sa, 128) : umma::desc_kmajor(sa, 128);
        const uint64_t bd0 = b_mn ? umma::desc_mnmajor(sb, 128) : umma::desc_kmajor(sb, 128);
        const uint64_t astep = a_mn ? 16u : 256u, bstep = b_mn ? 16u : 256u;
        uint32_t elected = 0;
        if (mode == 1) {
            asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.b32 %0, 1, 0, p;\n\t}\n" : "=r"(elected));
        } else {
            elected = ((tid & 31) == 0);
        }
        const uint32_t tbase = taddr + (nwarps > 1 ? 128 * warp : 0);
        t0 = clock64();
        if (uniform) {
            const uint32_t tb_u = __shfl_sync(0xffffffffu, tbase, 0);
            for (int r = 0; r < reps; ++r) {
                uint64_t ad = ad0, bd = bd0;
#pragma unroll 4
                for (int ks = 0; ks < ksteps; ++ks) {
                    for (int ac = 0; ac < nacc; ++ac) umma::mma_f16_elect(tb_u + (uint32_t)(ac * N), ad, bd, idesc, 1u);
                    ad += astep; bd += bstep;
                }
            }
            __syncwarp();
            t1 = clock64();
            umma::mma_commit_elect(&mbar);
            elected = 0;
        } else if (elected) {
            for (int r = 0; r < reps; ++r) {
                uint64_t ad = ad0, bd = bd0;
                for (int ks = 0; ks < ksteps; ++ks) {
                    for (int ac = 0; ac < nacc; ++ac) umma::mma_f16(tbase + (uint32_t)(ac * N), ad, bd, idesc, true);
                    ad += astep; bd += bstep;
                }
            }
        }
        __syncwarp();
        if (!uniform) t1 = clock64();
        if (elected) umma::mma_commit(&mbar);
        __syncwarp();
        ok = umma::mbar_wait(&mbar, 0);
        t2 = clock64();
        if (tid == 0) {
            cycles[0] = t1 - t0;
            cycles[1] = t2 - t0;
            *status = ok ? 0 : 1;
        }
    }
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 0) umma::tmem_dealloc(taddr, 512);
}
}  // namespace ddrl

extern "C" int ddrl_umma_bench(int M, int N, int a_mn, int b_mn, int reps, int ksteps, void* cycles2, int* status, void* stream) {
    DDRL_REQUIRE((M == 64 || M == 128) && N >= 8 && N <= 256 && N % 8 == 0 && reps >= 1 && (ksteps & 255) >= 1 && (ksteps & 255) <= 8 && cycles2 && status,
                 DDRL_E_BADARG, "umma_bench: bad arguments");
    static bool attr = false;
    if (!attr) {
        cudaFuncSetAttribute(ddrl::umma_bench_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);
        attr = true;
    }
    ddrl::umma_bench_kernel<<<1, 128, 96 * 1024, (cudaStream_t)stream>>>(M, N, a_mn, b_mn, reps, ksteps, (long long*)cycles2, status);
    DDRL_CHECK_LAUNCH("umma_bench");
    return DDRL_OK;
}

// =================================================================================================================
// Tensor-core FCNet training step: same contract as fcnet_train_kernel (csrc/fcnet.cu) — one minibatch of all
// policies, fused forward + PPO loss + backward, per-CTA partial gradients in flat checkpoint order — with every
// GEMM (layers, heads, head back-projection, all weight gradients) on tcgen05 (kind::f16, FP32 accumulation in TMEM).
// FP32 operands are split into fp16 (hi, lo) pairs and three products hi*hi + hi*lo + lo*hi are accumulated, which
// restores ~2^-21 relative accuracy (umma self test).
//
//   * tile = 128 rows (UMMA M); 512 threads, thread = (row, 16-column quarter) of a 64-wide branch tile, so a
//     tcgen05.ld 32x32b.x8 hands each thread 8 of its accumulators at a time; epilogues are short ROLLED loops over
//     8-column chunks (the previous fully unrolled version was 240 KB of SASS and instruction-fetch bound).
//   * the value and policy branches are processed one after the other (the PPO loss separates into a policy part
//     and a value part), which halves the activation footprint: H1, H2 are [128][64] fp16 hi/lo in the chunked layout.
//   * the SAME activation buffers feed the forward chain (K-major view) and the weight-gradient GEMMs (MN-major
//     view: M = feature, K = row), so the backward needs no transposed copies; weight gradients accumulate in TMEM
//     (M = 64 accumulators, row m in lane 32*(m/16) + m%16) across all tiles of the CTA.
//   * activations needed again by the backward (1 - h^2) are re-read from their hi + lo halves (exact to 2^-22).
//   * bias gradients ride along: X carries a constant-1 pad column, so dW1 gains a row = sum_r dz1 and a 16-wide
//     MMA against that column gives sum_r dz2.
//   * operands are stored pre-multiplied by power-of-two scales (exact) so the lo halves stay in the fp16 normal range;
//     loss gradients are kept without the 1/minibatch factor on chip; both are undone at the accumulator read-out.
//     fp16 overflow is clamped AND reported (*status = 2) so the caller can redo the step on the FP32 kernel.
// =================================================================================================================
#include "tc_common.cuh"

namespace ddrl {

// TMEM columns
constexpr int TC_DACC = 0, TC_HOUT = 64, TC_GW2 = 96, TC_GW1 = 224, TC_GB2 = 352, TC_GWH = 384, TC_TMEM_COLS = 512;

// Forward epilogue of this thread's 16 columns: act = tanh(acc * inv_in + bias) -> fp16 hi/lo (x TC_SH), chunked [128][64].
__device__ __noinline__ bool tc_epi_tanh(uint32_t taddr, const float* bias, float inv_in, unsigned char* dhi, unsigned char* dlo,
                                         int row, int cq) {
    bool ovf = false;
#pragma unroll 1
    for (int c = 0; c < 2; ++c) {
        float v[8];
        umma::tmem_ld8(taddr + 8 * c, v);
        const float4 b0 = *reinterpret_cast<const float4*>(bias + 8 * c);
        const float4 b1 = *reinterpret_cast<const float4*>(bias + 8 * c + 4);
        v[0] = tanhf(fmaf(v[0], inv_in, b0.x)); v[1] = tanhf(fmaf(v[1], inv_in, b0.y));
        v[2] = tanhf(fmaf(v[2], inv_in, b0.z)); v[3] = tanhf(fmaf(v[3], inv_in, b0.w));
        v[4] = tanhf(fmaf(v[4], inv_in, b1.x)); v[5] = tanhf(fmaf(v[5], inv_in, b1.y));
        v[6] = tanhf(fmaf(v[6], inv_in, b1.z)); v[7] = tanhf(fmaf(v[7], inv_in, b1.w));
        uint4 hi, lo;
        ovf = tc_split8(v, TC_SH, hi, lo) || ovf;
        const int off = ((2 * cq + c) * TC_ROWS + row) * 16;
        *reinterpret_cast<uint4*>(dhi + off) = hi;
        *reinterpret_cast<uint4*>(dlo + off) = lo;
    }
    return ovf;
}

// Backward epilogue: g = acc * inv_in * (1 - h^2), h re-read from the buffer it then overwrites (fp16 hi/lo x out_scale).
__device__ __noinline__ bool tc_epi_grad(uint32_t taddr, float inv_in, float out_scale, unsigned char* bhi, unsigned char* blo,
                                         int row, int cq) {
    bool ovf = false;
#pragma unroll 1
    for (int c = 0; c < 2; ++c) {
        float v[8], h[8];
        umma::tmem_ld8(taddr + 8 * c, v);
        const int off = ((2 * cq + c) * TC_ROWS + row) * 16;
        tc_join8(*reinterpret_cast<const uint4*>(bhi + off), *reinterpret_cast<const uint4*>(blo + off), 1.f / TC_SH, h);
#pragma unroll
        for (int j = 0; j < 8; ++j) v[j] = v[j] * inv_in * (1.f - h[j] * h[j]);
        uint4 hi, lo;
        ovf = tc_split8(v, out_scale, hi, lo) || ovf;
        *reinterpret_cast<uint4*>(bhi + off) = hi;
        *reinterpret_cast<uint4*>(blo + off) = lo;
    }
    return ovf;
}

template <int A>
__global__ void __launch_bounds__(TC_NT, 1) fcnet_train_tc_kernel(const TcTrainArgs a) {
    constexpr int A2 = 2 * A;
    extern __shared__ __align__(1024) unsigned char sm[];
    const int p = blockIdx.y, G = gridDim.x, bx = blockIdx.x;
    const int D = a.D, KX = tc_kx(D);
    const TcImg I = tc_img(D, A);
    const TcSmem S = tc_smem(D, A);
    const FcOffsets o = fc_offsets(D, A);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, q = warp & 3, cq = warp >> 2, row = q * 32 + lane;
    uint64_t* mbar = reinterpret_cast<uint64_t*>(sm + S.bar);
    uint32_t* tslot = reinterpret_cast<uint32_t*>(sm + S.bar + 8);
    const uint32_t sbase = umma::smem_u32(sm);

    const int step = a.step_ctr ? *a.step_ctr : 0;
    const int mb = a.mb_perm ? a.mb_perm[(int64_t)p * a.perm_stride + step] : step;
    const int64_t mb0 = (int64_t)mb * a.MB;
    const int64_t mb1 = min(mb0 + a.MB, a.R);
    const int rpc = (((a.MB + G - 1) / G) + 7) & ~7;
    const int64_t cr0 = min(mb0 + (int64_t)bx * rpc, mb1), cr1 = min(cr0 + rpc, mb1);
    const int NPs = (o.NP + 3) & ~3;
    float* gp = a.grad_part + ((int64_t)p * G + bx) * NPs;
    do {   // single exit towards the fused tail (one inlined copy of it)
    if (cr1 <= cr0) {   // no rows: zero partial, no tensor work (still takes part in the fused tail)
        for (int i = tid; i < o.NP; i += TC_NT) gp[i] = 0.f;
        if (tid < DDRL_NSTAT && a.stat_part) a.stat_part[((int64_t)p * G + bx) * DDRL_NSTAT + tid] = 0.0;
        break;
    }

    const float* obs_p = a.obs + (int64_t)p * a.R * D;
    float* xraw = reinterpret_cast<float*>(sm + S.xraw);
    float* pf = reinterpret_cast<float*>(sm + S.pf);
    const float* b1c = reinterpret_cast<const float*>(sm + I.b1c);
    const float* b2c = reinterpret_cast<const float*>(sm + I.b2c);
    const float* sbo = reinterpret_cast<const float*>(sm + I.bo);
    const float* sbvo = reinterpret_cast<const float*>(sm + I.bvo);

    auto prefetch_x = [&](int64_t r0, int n) {
        for (int i = tid; i < n * D; i += TC_NT) tc_cp4(xraw + i, obs_p + r0 * D + i);
    };
    auto prefetch_loss = [&](int64_t r0, int n) {
        const int64_t g0 = (int64_t)p * a.R + r0;
        float* pa = pf;
        float* po = pa + TC_ROWS * A;
        float* ps = po + TC_ROWS * A2;
        for (int i = tid; i < n * A; i += TC_NT) tc_cp4(pa + i, a.actions + g0 * A + i);
        for (int i = tid; i < n * A2; i += TC_NT) tc_cp4(po + i, a.old_logits + g0 * A2 + i);
        for (int i = tid; i < n; i += TC_NT) {
            tc_cp4(ps + i, a.old_logp + g0 + i);
            tc_cp4(ps + TC_ROWS + i, a.vf_preds + g0 + i);
            tc_cp4(ps + 2 * TC_ROWS + i, a.adv + g0 + i);
            tc_cp4(ps + 3 * TC_ROWS + i, a.vtarg + g0 + i);
        }
    };

    // ---- setup: TMEM, mbarrier, weights image, first tile's inputs ------------------------------------------------
    if (warp == 0) umma::tmem_alloc(tslot, TC_TMEM_COLS);
    if (tid == 0) { umma::mbar_init(mbar, 1); umma::fence_mbar_init(); }
    {
        const unsigned char* img_p = a.img + (int64_t)p * I.bytes;
        for (int i = tid; i < I.bytes / 16; i += TC_NT) tc_cp16(sm + 16 * i, img_p + 16 * i);
        const int n0 = (int)min((int64_t)TC_ROWS, cr1 - cr0);
        prefetch_x(cr0, n0);
        prefetch_loss(cr0, n0);
        asm volatile("cp.async.commit_group;\n" ::);
    }
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = *tslot;
    const uint32_t tlane = (uint32_t)(q * 32) << 16;
    uint32_t phase = 0;
    bool ok = true, first = true;
    int ovf = 0;   // bit mask of fp16 overflows: 2 = x, 4 = activations, 8 = dl, 16 = dz2, 32 = dz1
    const float klc = a.kl_coeff[p];
    double st[DDRL_NSTAT];
#pragma unroll
    for (int i = 0; i < DDRL_NSTAT; ++i) st[i] = 0.0;
    float gbh[A2 + 1];   // head bias gradients (loss threads): sum_r dl[r][o]
#pragma unroll
    for (int i = 0; i < A2 + 1; ++i) gbh[i] = 0.f;
    const int ch0 = (D >> 3) & ~1;     // 16-column window of X that contains the constant-1 pad column D

    auto wait_mma = [&]() {
        ok = umma::mbar_wait(mbar, phase) && ok;
        phase ^= 1;
        umma::fence_after_sync();
    };
    auto publish = [&]() {   // generic smem writes -> async proxy, TMEM reads retired, then CTA barrier
        umma::fence_async_smem();
        umma::fence_before_sync();
        __syncthreads();
    };

#pragma unroll 1
    for (int64_t row0 = cr0; row0 < cr1; row0 += TC_ROWS) {
        const int nrows = (int)min((int64_t)TC_ROWS, cr1 - row0);
        asm volatile("cp.async.wait_group 0;\n" ::: "memory");
        __syncthreads();
        // ---- x: fp32 staging -> fp16 hi/lo chunked [128][KX], constant 1 in column D, zero rows beyond nrows ----------
        {
            const int r = tid & (TC_ROWS - 1);
#pragma unroll 1
            for (int c8 = tid >> 7; c8 < (KX >> 3); c8 += 4) {
                float v[8];
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    const int d = c8 * 8 + e;
                    v[e] = (r < nrows) ? (d < D ? xraw[r * D + d] : (d == D ? 1.f : 0.f)) : 0.f;
                }
                uint4 hi, lo;
                ovf |= tc_split8(v, TC_SX, hi, lo) ? 2 : 0;
                *reinterpret_cast<uint4*>(sm + S.X[0] + (c8 * TC_ROWS + r) * 16) = hi;
                *reinterpret_cast<uint4*>(sm + S.X[1] + (c8 * TC_ROWS + r) * 16) = lo;
            }
        }
        publish();
        {   // staging buffer is free again: stream in the next tile's observations behind this tile's compute
            const int64_t nxt = row0 + TC_ROWS;
            if (nxt < cr1) prefetch_x(nxt, (int)min((int64_t)TC_ROWS, cr1 - nxt));
            asm volatile("cp.async.commit_group;\n" ::);
        }

#pragma unroll 1
        for (int bi = 0; bi < 2; ++bi) {
            const int b = 1 - bi;                      // value branch first, then policy
            const uint32_t dacc = tmem + tlane + TC_DACC + 16 * cq;
            // ---- F1: Dacc = X * W1b^T ------------------------------------------------------------------------
            if (tid == 0) {
                umma::fence_after_sync();
                tc_gemm(tmem + TC_DACC, sbase + S.X[0], sbase + S.X[1], TC_ROWS, false, sbase + I.W1[b][0],
                        sbase + I.W1[b][1], 64, false, 128, 64, KX >> 4, false, 3);
                umma::mma_commit(mbar);
            }
            wait_mma();
            ovf |= tc_epi_tanh(dacc, b1c + b * 64 + 16 * cq, 1.f / (TC_SX * TC_SW), sm + S.H1[0], sm + S.H1[1], row, cq) ? 4 : 0;
            publish();
            // ---- F2: Dacc = H1 * W2b ---------------------------------------------------------------------------
            if (tid == 0) {
                umma::fence_after_sync();
                tc_gemm(tmem + TC_DACC, sbase + S.H1[0], sbase + S.H1[1], TC_ROWS, false, sbase + I.W2[b][0],
                        sbase + I.W2[b][1], 64, true, 128, 64, 4, false, 3);
                umma::mma_commit(mbar);
            }
            wait_mma();
            ovf |= tc_epi_tanh(dacc, b2c + b * 64 + 16 * cq, 1.f / (TC_SH * TC_SW), sm + S.H2[0], sm + S.H2[1], row, cq) ? 4 : 0;
            publish();
            // ---- heads: Hout[128][16] = H2 * WoT_b^T ---------------------------------------------------------------
            if (tid == 0) {
                umma::fence_after_sync();
                tc_gemm(tmem + TC_HOUT, sbase + S.H2[0], sbase + S.H2[1], TC_ROWS, false, sbase + I.WoT[b][0],
                        sbase + I.WoT[b][1], TC_NO, false, 128, TC_NO, 4, false, 3);
                umma::mma_commit(mbar);
            }
            wait_mma();
            // ---- loss of this branch (warps 0..3, one thread per row) -> DL (fp16 hi/lo x TC_SL, chunked [128][16]) ------
            if (cq == 0) {
                float out[16], dl[16];
                umma::tmem_ld16(tmem + tlane + TC_HOUT, out);
                double s[DDRL_NSTAT];
#pragma unroll
                for (int i = 0; i < DDRL_NSTAT; ++i) s[i] = 0.0;
#pragma unroll
                for (int i = 0; i < 16; ++i) dl[i] = 0.f;
                if (row < nrows) {
                    const float* pa = pf;
                    const float* po = pa + TC_ROWS * A;
                    const float* ps = po + TC_ROWS * A2;
                    if (b == 0) {
                        float lg[A2];
#pragma unroll
                        for (int oo = 0; oo < A2; ++oo) lg[oo] = fmaf(out[oo], 1.f / (TC_SH * TC_SW), sbo[oo]);
                        ppo_row_policy(lg, A, pa + row * A, po + row * A2, ps[row], ps[2 * TC_ROWS + row], klc,
                                       a.hp.clip_param, a.hp.entropy_coeff, 1.f, dl, s);
#pragma unroll
                        for (int oo = 0; oo < A2; ++oo) gbh[oo] += dl[oo];
                    } else {
                        const float val = fmaf(out[0], 1.f / (TC_SH * TC_SW), sbvo[0]);
                        dl[0] = ppo_row_value(val, ps[TC_ROWS + row], ps[3 * TC_ROWS + row], a.hp.vf_clip_param,
                                              a.hp.vf_loss_coeff, 1.f, s);
                        gbh[A2] += dl[0];
                    }
                }
                if (first) {   // per-branch gradient scale of this CTA: power of two with max|dl| * scale ~ TC_GTARGET
                    float mx = 0.f;
#pragma unroll
                    for (int i = 0; i < 16; ++i) mx = fmaxf(mx, fabsf(dl[i]));
#pragma unroll
                    for (int off = 16; off > 0; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
                    float* smx = reinterpret_cast<float*>(sm + S.red);
                    if (lane == 0) smx[warp] = mx;
                    asm volatile("bar.sync 1, 128;" ::: "memory");     // the four loss warps only
                    mx = fmaxf(fmaxf(smx[0], smx[1]), fmaxf(smx[2], smx[3]));
                    int e = 0;
                    if (mx > 0.f && mx < 3.0e38f) e = (int)floorf(log2f(TC_GTARGET / mx));
                    e = max(-20, min(20, e));
                    if (tid == 0) reinterpret_cast<float*>(sm + S.bar + 16)[b] = exp2f((float)e);
                    asm volatile("bar.sync 1, 128;" ::: "memory");
                }
                const float sg_l = reinterpret_cast<const float*>(sm + S.bar + 16)[b];
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                    uint4 hi, lo;
                    ovf |= tc_split8(&dl[8 * c], sg_l, hi, lo) ? 8 : 0;
                    *reinterpret_cast<uint4*>(sm + S.DL[0] + (c * TC_ROWS + row) * 16) = hi;
                    *reinterpret_cast<uint4*>(sm + S.DL[1] + (c * TC_ROWS + row) * 16) = lo;
                }
#pragma unroll
                for (int i = 0; i < DDRL_NSTAT; ++i) st[i] += s[i];
            }
            publish();
            const float sg = reinterpret_cast<const float*>(sm + S.bar + 16)[b];   // this branch's gradient scale
            // ---- B1: gWh_b[k][o] (+)= H2^T DL ;  dz2-pre: Dacc = DL * WoT_b (B MN-major: N = hidden unit, K = output) ----
            if (tid == 0) {
                umma::fence_after_sync();
                tc_gemm(tmem + TC_GWH + 16 * b, sbase + S.H2[0], sbase + S.H2[1], TC_ROWS, true, sbase + S.DL[0],
                        sbase + S.DL[1], TC_ROWS, true, 64, 16, 8, !first, 3);
                tc_gemm(tmem + TC_DACC, sbase + S.DL[0], sbase + S.DL[1], TC_ROWS, false, sbase + I.WoT[b][0],
                        sbase + I.WoT[b][1], TC_NO, true, 128, 64, 1, false, 3);
                umma::mma_commit(mbar);
            }
            wait_mma();      // B1 has consumed H2; dz2 = pre * (1 - h2^2) overwrites it
            ovf |= tc_epi_grad(dacc, 1.f / (sg * TC_SW), sg, sm + S.H2[0], sm + S.H2[1], row, cq) ? 16 : 0;
            publish();
            // ---- B3: gW2_b (+)= H1^T dZ2;  gb2_b (+)= dZ2^T 1;  B4: Dacc = dZ2 * W2b^T -------------------------------
            if (tid == 0) {
                umma::fence_after_sync();
                tc_gemm(tmem + TC_GW2 + 64 * b, sbase + S.H1[0], sbase + S.H1[1], TC_ROWS, true, sbase + S.H2[0],
                        sbase + S.H2[1], TC_ROWS, true, 64, 64, 8, !first, 3);
                tc_gemm(tmem + TC_GB2 + 16 * b, sbase + S.H2[0], sbase + S.H2[1], TC_ROWS, true,
                        sbase + S.X[0] + ch0 * TC_ROWS * 16, 0, TC_ROWS, true, 64, 16, 8, !first, 2);
                tc_gemm(tmem + TC_DACC, sbase + S.H2[0], sbase + S.H2[1], TC_ROWS, false, sbase + I.W2[b][0],
                        sbase + I.W2[b][1], 64, false, 128, 64, 4, false, 3);
                umma::mma_commit(mbar);
            }
            wait_mma();      // B3 has consumed H1; dz1 = (dz2 W2^T) * (1 - h1^2) overwrites it
            ovf |= tc_epi_grad(dacc, 1.f / (sg * TC_SW), sg, sm + S.H1[0], sm + S.H1[1], row, cq) ? 32 : 0;
            publish();
            // ---- B5: gW1_b[c][d] (+)= dZ1^T X   (column D of X is the constant 1 -> bias gradient) ------------------
            if (tid == 0) {
                umma::fence_after_sync();
                tc_gemm(tmem + TC_GW1 + 64 * b, sbase + S.H1[0], sbase + S.H1[1], TC_ROWS, true, sbase + S.X[0],
                        sbase + S.X[1], TC_ROWS, true, 64, KX, 8, !first, 3);
                if (bi == 1) umma::mma_commit(mbar);   // first branch: committed together with the next branch's F1
            }
            if (bi == 1) wait_mma();
        }
        {   // both branches consumed the staged loss inputs: fetch the next tile's
            const int64_t nxt = row0 + TC_ROWS;
            if (nxt < cr1) prefetch_loss(nxt, (int)min((int64_t)TC_ROWS, cr1 - nxt));
            asm volatile("cp.async.commit_group;\n" ::);
        }
        first = false;
    }
    asm volatile("cp.async.wait_group 0;\n" ::: "memory");

    // ---- write-out: TMEM accumulators (M = 64: row m lives in lane 32*(m/16) + m%16) -> flat partial, x 1/minibatch ----
    const float inv = a.hp.inv_global_mb;
    __syncthreads();
    const int m = 16 * q + lane;            // valid for lane < 16
    const bool mine = lane < 16;
#pragma unroll 1
    for (int b = 0; b < 2; ++b) {
        float v[8];
        const float sgb = reinterpret_cast<const float*>(sm + S.bar + 16)[b];
        const float inv_gw2 = inv / (TC_SH * sgb), inv_gw1 = inv / (sgb * TC_SX), inv_gwh = inv_gw2;
#pragma unroll 1
        for (int c = 0; c < 2; ++c) {        // gW2_b: this warp's 16 columns
            umma::tmem_ld8(tmem + tlane + TC_GW2 + 64 * b + 16 * cq + 8 * c, v);
            if (mine) {
                float* dst = gp + (b ? o.Wv2 : o.W2) + m * 64 + 16 * cq + 8 * c;
#pragma unroll
                for (int j = 0; j < 8; ++j) dst[j] = v[j] * inv_gw2;
            }
        }
#pragma unroll 1
        for (int c8 = cq; c8 < (KX >> 3); c8 += 4) {   // gW1_b[c = m][d]: 8 input features at a time
            umma::tmem_ld8(tmem + tlane + TC_GW1 + 64 * b + 8 * c8, v);
            if (mine) {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int d = 8 * c8 + j;
                    if (d < D) gp[(b ? o.Wv1 : o.W1) + d * 64 + m] = v[j] * inv_gw1;
                    else if (d == D) gp[(b ? o.bv1 : o.b1) + m] = v[j] * inv_gw1;
                }
            }
        }
        if (cq == 0) {                                   // gb2_b: column of the constant-1 pad inside its 16-wide window
            umma::tmem_ld8(tmem + tlane + TC_GB2 + 16 * b + (((D - 8 * ch0) >> 3) << 3), v);
            const int jsel = (D - 8 * ch0) & 7;
            const float g = jsel == 0 ? v[0] : jsel == 1 ? v[1] : jsel == 2 ? v[2] : jsel == 3 ? v[3] : jsel == 4 ? v[4]
                          : jsel == 5 ? v[5] : jsel == 6 ? v[6] : v[7];
            if (mine) gp[(b ? o.bv2 : o.b2) + m] = g * inv_gw1;
        }
        if (cq == 1) {                                   // gWh_b[k = m][o]
            float w[16];
            umma::tmem_ld16(tmem + tlane + TC_GWH + 16 * b, w);
            if (mine) {
                if (b == 0) {
#pragma unroll
                    for (int oo = 0; oo < A2; ++oo) gp[o.Wo + m * A2 + oo] = w[oo] * inv_gwh;
                } else {
                    gp[o.Wvo + m] = w[0] * inv_gwh;
                }
            }
        }
    }
    // head bias gradients and stats: reduce over the 128 loss threads (warps 0..3), fixed order
    __syncthreads();
    double* redd = reinterpret_cast<double*>(sm + S.red);          // [4 warps][32]
    if (cq == 0) {
#pragma unroll
        for (int i = 0; i < A2 + 1; ++i) {
            const float s = warp_sum(gbh[i]);
            if (lane == 0) redd[warp * 32 + 8 + i] = (double)s;
        }
#pragma unroll
        for (int i = 0; i < DDRL_NSTAT; ++i) {
            const double s = warp_sum(st[i]);
            if (lane == 0) redd[warp * 32 + i] = s;
        }
    }
    __syncthreads();
    if (tid <= A2) {
        const float s = (float)((redd[8 + tid] + redd[32 + 8 + tid]) + (redd[64 + 8 + tid] + redd[96 + 8 + tid])) * inv;
        gp[tid == A2 ? o.bvo : o.bo + tid] = s;
    }
    if (tid < DDRL_NSTAT && a.stat_part)
        a.stat_part[((int64_t)p * G + bx) * DDRL_NSTAT + tid] = (redd[tid] + redd[32 + tid]) + (redd[64 + tid] + redd[96 + tid]);
    if (a.status) {
        if (tid == 0 && !ok) atomicOr(a.status, 1);
        if (ovf) atomicOr(a.status, ovf);
    }
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 0) umma::tmem_dealloc(tmem, TC_TMEM_COLS);
    } while (0);
    if (a.tail.theta) {   // fused grad-reduce + clip + Adam (single-GPU SGD loop)
        const bool tok = sgd_step_tail(a.tail, tail_single_step(a.tail, p), a.grad_part, a.stat_part, p, gridDim.y, bx, G, o.NP, step, D, A,
                                       reinterpret_cast<float*>(sm + S.H1[0]));
        if (!tok && tid == 0 && a.status) atomicOr(a.status, 64);
    }
}

// flat theta -> tensor-core image (fp16 hi/lo of 256*w for the GEMM weights + fp32 biases)
__global__ void fcnet_tc_pack_kernel(const float* __restrict__ theta, int D, int A, unsigned char* __restrict__ img) {
    const int p = blockIdx.y;
    const TcImg L = tc_img(D, A);
    const FcOffsets o = fc_offsets(D, A);
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= o.NP) return;
    bool f16;
    int p0, p1;
    tc_img_pos(L, o, D, A, j, f16, p0, p1);
    const float w = theta[(int64_t)p * o.NP + j];
    unsigned char* im = img + (int64_t)p * L.bytes;
    if (f16) {
        __half hi, lo;
        umma::split_f16(w * TC_SW, hi, lo);
        *reinterpret_cast<__half*>(im + p0) = hi;
        *reinterpret_cast<__half*>(im + p1) = lo;
    } else {
        *reinterpret_cast<float*>(im + p0) = w;
    }
}

}  // namespace ddrl

extern "C" int ddrl_fcnet_tc_image_bytes(int D, int A) {
    if (D < 1 || D > DDRL_MAX_OBS - 1 || !(A == 1 || A == 2 || A == 4 || A == 8)) return DDRL_E_UNSUPPORTED_SHAPE;
    return tc_img(D, A).bytes;
}

extern "C" int ddrl_fcnet_tc_pack(const float* theta, int P, int D, int A, void* img, void* stream) {
    DDRL_REQUIRE(theta && img && P >= 1, DDRL_E_BADARG, "fcnet_tc_pack: null pointer or bad P");
    DDRL_REQUIRE(D >= 1 && D <= DDRL_MAX_OBS - 1 && (A == 1 || A == 2 || A == 4 || A == 8), DDRL_E_UNSUPPORTED_SHAPE,
                 "fcnet_tc_pack: unsupported D=%d A=%d (A in {1,2,4,8}, D <= 63)", D, A);
    const int NP = fc_offsets(D, A).NP;
    cudaMemsetAsync(img, 0, (size_t)P * tc_img(D, A).bytes, (cudaStream_t)stream);
    fcnet_tc_pack_kernel<<<dim3((NP + 255) / 256, P), 256, 0, (cudaStream_t)stream>>>(theta, D, A, (unsigned char*)img);
    DDRL_CHECK_LAUNCH("fcnet_tc_pack");
    return DDRL_OK;
}

static int g_tc_variant = 0;   // 0 = automatic, 1 = branch-sequential kernel, 2 = ping-pong kernel
static long long* g_tc_dbg_clock = nullptr;

extern "C" int ddrl_tc_pingpong_eligible(int D, int A) {
    if (D < 1 || D > DDRL_MAX_OBS - 1 || !(A == 1 || A == 2 || A == 4 || A == 8)) return 0;
    return (g_tc_variant != 1 && tc2_eligible(D, A)) ? 1 : 0;
}

extern "C" int ddrl_tc_set_debug_clock(void* device_int64x64) {
    g_tc_dbg_clock = reinterpret_cast<long long*>(device_int64x64);
    return DDRL_OK;
}

extern "C" int ddrl_tc_set_variant(int variant) {
    DDRL_REQUIRE(variant >= 0 && variant <= 2, DDRL_E_BADARG, "tc_set_variant: variant must be 0, 1 or 2");
    g_tc_variant = variant;
    return DDRL_OK;
}

template <int A>
static int launch_tc(const TcTrainArgs& a, int P, int G, size_t smem, cudaStream_t st) {
    if (int rc = raise_smem_once<fcnet_train_tc_kernel<A>>("ppo_train_step_tc")) return rc;
    fcnet_train_tc_kernel<A><<<dim3(G, P), TC_NT, smem, st>>>(a);
    return DDRL_OK;
}

// What the two tensor-core train steps share: the pointer and P/R/MB/ctas check, then the entry's own checks
// (`entry_checks`), the weight-image alignment, the fused-tail check, and the TcTrainArgs fields (dbg_clock stays null).
// `pingpong`: the step runs on the ping-pong kernel (the only one that can keep the accumulation vector, launch_tail).
template <class EntryChecks>
static int tc_train_args(TcTrainArgs& a, const char* who, bool entry_ptrs, EntryChecks&& entry_checks, bool pingpong,
                         const void* tc_img_p, const float* obs, const float* actions, const float* old_logits,
                         const float* old_logp, const float* vf_preds, const float* adv, const float* vtarg, int P, int64_t R,
                         int D, int A, int MB, const int32_t* mb_perm, int64_t perm_stride, const int32_t* step_ctr,
                         const float* kl_coeff, const ddrl_ppo_hyper* hyper, int ctas_per_policy, float* grad_part,
                         double* stat_part, int* status, const ddrl_sgd_tail* tail) {
    DDRL_REQUIRE(entry_ptrs && tc_img_p && obs && actions && old_logits && old_logp && vf_preds && adv && vtarg && kl_coeff &&
                     hyper && grad_part && P >= 1 && R >= 1 && MB >= 1 && ctas_per_policy >= 1,
                 DDRL_E_BADARG, "%s: null pointer or bad P/R/MB/ctas", who);
    if (int rc = entry_checks()) return rc;
    DDRL_REQUIRE((reinterpret_cast<uintptr_t>(tc_img_p) & 15) == 0, DDRL_E_BADARG,
                 "%s: the weight image must be 16-byte aligned (TMA bulk copies)", who);
    if (tail)
        if (int rc = sgd_tail_check(tail, ctas_per_policy * P, who)) return rc;
    a = TcTrainArgs{};
    a.img = (const unsigned char*)tc_img_p; a.obs = obs; a.actions = actions; a.old_logits = old_logits;
    a.old_logp = old_logp; a.vf_preds = vf_preds; a.adv = adv; a.vtarg = vtarg; a.R = R; a.D = D; a.A = A; a.MB = MB;
    a.mb_perm = mb_perm; a.perm_stride = perm_stride; a.step_ctr = step_ctr; a.kl_coeff = kl_coeff; a.hp = *hyper;
    a.grad_part = grad_part; a.stat_part = stat_part; a.status = status;
    a.tail = launch_tail(tail, pingpong && !tc2_clusters_requested());
    return DDRL_OK;
}

extern "C" int ddrl_ppo_train_step_tc(const void* tc_img_p, const float* obs, const float* actions, const float* old_logits,
                                      const float* old_logp, const float* vf_preds, const float* adv, const float* vtarg,
                                      int P, int64_t R, int D, int A, int MB, const int32_t* mb_perm, int64_t perm_stride,
                                      const int32_t* step_ctr, const float* kl_coeff, const ddrl_ppo_hyper* hyper,
                                      int ctas_per_policy, float* grad_part, double* stat_part, int* status,
                                      const ddrl_sgd_tail* tail, void* stream) {
    const char* who = "ppo_train_step_tc";
    const bool pingpong = g_tc_variant == 2 || (g_tc_variant == 0 && tc2_eligible(D, A));
    TcTrainArgs a;
    const int rc = tc_train_args(
        a, who, true,
        [&]() -> int {
            DDRL_REQUIRE(D >= 1 && D <= DDRL_MAX_OBS - 1 && (A == 1 || A == 2 || A == 4 || A == 8), DDRL_E_UNSUPPORTED_SHAPE,
                         "ppo_train_step_tc: unsupported D=%d A=%d (A in {1,2,4,8}, D <= 63)", D, A);
            return DDRL_OK;
        },
        pingpong, tc_img_p, obs, actions, old_logits, old_logp, vf_preds, adv, vtarg, P, R, D, A, MB, mb_perm, perm_stride,
        step_ctr, kl_coeff, hyper, ctas_per_policy, grad_part, stat_part, status, tail);
    if (rc != DDRL_OK) return rc;
    a.dbg_clock = g_tc_dbg_clock;
    DDRL_REQUIRE(!tail || tail->nsteps <= 1 || pingpong, DDRL_E_UNSUPPORTED_SHAPE,
                 "ppo_train_step_tc: nsteps > 1 needs the ping-pong kernel (D <= 47)");
    const size_t smem = (size_t)tc_smem(D, A).total;
    DDRL_REQUIRE(smem <= 227 * 1024, DDRL_E_UNSUPPORTED_SHAPE, "ppo_train_step_tc: shared memory %zu > 227 KB", smem);
    int lrc;
    if (pingpong) {
        DDRL_REQUIRE(tc2_eligible(D, A), DDRL_E_UNSUPPORTED_SHAPE,
                     "ppo_train_step_tc: ping-pong variant needs D <= 47 (D=%d, A=%d)", D, A);
        lrc = launch_tc2(a, P, ctas_per_policy, (cudaStream_t)stream);
    } else {
        lrc = dispatch_A(A, "ppo_train_step_tc: unsupported A", [&](auto A_) {
            return launch_tc<decltype(A_)::value>(a, P, ctas_per_policy, smem, (cudaStream_t)stream);
        });
    }
    if (lrc != DDRL_OK) return lrc;
    DDRL_CHECK_LAUNCH(who);
    return DDRL_OK;
}

extern "C" int ddrl_ppo_train_step_tc_coupled(const void* tc_img_p, const float* theta, const int32_t* node_id, const float* obs,
                                              const float* actions, const float* old_logits, const float* old_logp,
                                              const float* vf_preds, const float* adv, const float* vtarg, int P, int64_t R,
                                              int D, int A, int MB, const int32_t* mb_perm, int64_t perm_stride,
                                              const int32_t* step_ctr, const float* kl_coeff, const ddrl_ppo_hyper* hyper,
                                              int ctas_per_policy, float* grad_part, double* stat_part, int* status,
                                              const ddrl_sgd_tail* tail, void* stream) {
    const char* who = "ppo_train_step_tc_coupled";
    TcTrainArgs a;
    const int rc = tc_train_args(
        a, who, theta && node_id,
        [&]() -> int {
            DDRL_REQUIRE(A == 2, DDRL_E_BADARG, "ppo_train_step_tc_coupled: LegCoupling needs A = 2 (num_outputs == 4), got A=%d", A);
            DDRL_REQUIRE(P == 1, DDRL_E_BADARG,
                         "ppo_train_step_tc_coupled: the coupled model is one shared policy (P = 1), got P=%d", P);
            DDRL_REQUIRE(D == 19 || D == 20, DDRL_E_UNSUPPORTED_SHAPE,
                         "ppo_train_step_tc_coupled: instantiated for SharedDecentralLegID (D = 19 or 20), got D=%d", D);
            DDRL_REQUIRE(tail != nullptr, DDRL_E_BADARG, "ppo_train_step_tc_coupled: the fused tail is required (NP + 8 parameters)");
            DDRL_REQUIRE(tail->theta == theta, DDRL_E_BADARG, "ppo_train_step_tc_coupled: tail->theta must be theta");
            DDRL_REQUIRE(status != nullptr, DDRL_E_BADARG,
                         "ppo_train_step_tc_coupled: status is required (it receives DDRL_STATUS_BAD_NODE for a node id outside 0..3)");
            DDRL_REQUIRE(!tail->ll_ws, DDRL_E_BADARG, "ppo_train_step_tc_coupled: the LL tail is not supported with leg coupling");
            DDRL_REQUIRE(g_tc_variant != 1, DDRL_E_BADARG,
                         "ppo_train_step_tc_coupled: only the ping-pong kernel has a coupled instantiation (ddrl_tc_set_variant(1) is set)");
            return DDRL_OK;
        },
        true, tc_img_p, obs, actions, old_logits, old_logp, vf_preds, adv, vtarg, P, R, D, A, MB, mb_perm, perm_stride,
        step_ctr, kl_coeff, hyper, ctas_per_policy, grad_part, stat_part, status, tail);
    if (rc != DDRL_OK) return rc;
    const int lrc = launch_tc2_cup(a, node_id, theta, P, ctas_per_policy, (cudaStream_t)stream);
    if (lrc != DDRL_OK) return lrc;
    DDRL_CHECK_LAUNCH(who);
    return DDRL_OK;
}

// The alignment check, TcTrainArgs and grid of the two tensor-core forwards: G CTAs per policy, at most sms / P of them.
static int tc_forward_args(TcTrainArgs& a, int& G, const char* who, const void* tc_img_p, const float* obs, const double* norm,
                           float clip, int P, int64_t R, int D, int A, float* obs_out, float* logits, float* value,
                           const float* eps, float* action, float* logp, int* status) {
    DDRL_REQUIRE(R <= 0x7fffffff, DDRL_E_UNSUPPORTED_SHAPE, "%s: R must fit 31 bits", who);
    DDRL_REQUIRE((reinterpret_cast<uintptr_t>(tc_img_p) & 15) == 0, DDRL_E_BADARG,
                 "%s: the weight image must be 16-byte aligned (TMA bulk copies)", who);
    a = TcTrainArgs{};
    a.img = (const unsigned char*)tc_img_p; a.obs = obs; a.R = R; a.D = D; a.A = A; a.MB = (int)R;
    a.hp = ddrl_ppo_hyper{0.f, 0.f, 0.f, 0.f, 1.f};
    a.status = status;
    a.norm = norm; a.clip = clip; a.obs_out = obs_out; a.logits_out = logits; a.value_out = value; a.eps = eps;
    a.action_out = action; a.logp_out = logp;
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    G = (int)std::max<int64_t>(1, std::min<int64_t>((R + TC_ROWS - 1) / TC_ROWS, std::max(1, sms / P)));
    return DDRL_OK;
}

extern "C" int ddrl_fcnet_forward_tc(const void* tc_img_p, const float* obs, const double* norm, float clip, int P, int64_t R,
                                     int D, int A, float* obs_out, float* logits, float* value, const float* eps, float* action,
                                     float* logp, int* status, void* stream) {
    DDRL_REQUIRE(tc_img_p && obs && P >= 1 && R >= 0, DDRL_E_BADARG, "fcnet_forward_tc: null pointer or bad P/R");
    DDRL_REQUIRE(!eps || (action && logp), DDRL_E_BADARG, "fcnet_forward_tc: eps given without action / logp outputs");
    DDRL_REQUIRE(D >= 1 && D <= DDRL_MAX_OBS - 1 && (A == 1 || A == 2 || A == 4 || A == 8) && tc2_eligible(D, A),
                 DDRL_E_UNSUPPORTED_SHAPE, "fcnet_forward_tc: unsupported D=%d A=%d (A in {1,2,4,8}, D <= 47)", D, A);
    if (R == 0) return DDRL_OK;
    TcTrainArgs a;
    int G = 0;
    int rc = tc_forward_args(a, G, "fcnet_forward_tc", tc_img_p, obs, norm, clip, P, R, D, A, obs_out, logits, value, eps,
                             action, logp, status);
    if (rc != DDRL_OK) return rc;
    rc = launch_tc2_forward(a, P, G, (cudaStream_t)stream);
    if (rc != DDRL_OK) return rc;
    DDRL_CHECK_LAUNCH("fcnet_forward_tc");
    return DDRL_OK;
}

extern "C" int ddrl_fcnet_forward_tc_coupled(const void* tc_img_p, const int32_t* node_id, const float* coupling, const float* obs,
                                             const double* norm, float clip, int P, int64_t R, int D, int A, float* obs_out,
                                             float* logits, float* value, const float* eps, float* action, float* logp, int* status,
                                             void* stream) {
    DDRL_REQUIRE(tc_img_p && node_id && coupling && obs && status && R >= 0, DDRL_E_BADARG,
                 "fcnet_forward_tc_coupled: null tc_img/node_id/coupling/obs/status or bad R");
    DDRL_REQUIRE(A == 2, DDRL_E_BADARG, "fcnet_forward_tc_coupled: LegCoupling needs A = 2 (num_outputs == 4), got A=%d", A);
    DDRL_REQUIRE(P == 1, DDRL_E_BADARG, "fcnet_forward_tc_coupled: the coupled model is one shared policy (P = 1), got P=%d", P);
    DDRL_REQUIRE(!eps || (action && logp), DDRL_E_BADARG, "fcnet_forward_tc_coupled: eps given without action / logp outputs");
    DDRL_REQUIRE(D == 19 || D == 20, DDRL_E_UNSUPPORTED_SHAPE,
                 "fcnet_forward_tc_coupled: instantiated for SharedDecentralLegID (D = 19 or 20), got D=%d", D);
    TcTrainArgs a;
    int G = 0;
    int rc = tc_forward_args(a, G, "fcnet_forward_tc_coupled", tc_img_p, obs, norm, clip, P, R, D, A, obs_out, logits, value, eps,
                             action, logp, status);
    if (rc != DDRL_OK || R == 0) return rc;
    rc = launch_tc2_forward_cup(a, node_id, coupling, G, (cudaStream_t)stream);
    if (rc != DDRL_OK) return rc;
    DDRL_CHECK_LAUNCH("fcnet_forward_tc_coupled");
    return DDRL_OK;
}

// Fused tail of one SGD step, executed by the SAME kernel that produced the per-CTA partial gradients:
//
//   barrier A (the G CTAs of a policy)                      partials visible
//   slice reduce: CTA bx owns parameters [bx*S, bx*S+S) and sums them over the G partials — up to 8 thread groups load
//                 different partials concurrently (one L2 round trip instead of G dependent ones), fixed summation order
//   [world > 1]   in-kernel all-reduce over NVLink peer memory, low-latency ("LL") style: every reduced element is PUSHED
//                 into every rank's exchange buffer as a 64-bit word {value, sequence flag} (two words per 16-byte store)
//                 — no fence, no separate flag round trip — and the owner thread polls its own buffer until the `world` words carry this step's
//                 sequence number, then adds them in rank order.  Every rank ends with bit-identical sums after one
//                 NVLink one-way latency; no NCCL call, no extra launch.  Buffers alternate by step parity.
//   barrier B     per-slice ||g||^2 visible -> global norm (same order everywhere), tf.clip_by_global_norm, TF1 Adam on
//                 the slice, packed weight images kept in step
//   ticket        the last CTA of the grid advances beta powers / step counter / exchange sequence and re-arms barriers
//
// It replaces grad_reduce + [ncclAllReduce] + clip_adam (two or three launches and their gaps per step).  All CTAs of the
// grid must be co-resident (callers launch at most one CTA per SM); every spin is bounded and reports instead of hanging.
#pragma once
#include <cuda_fp16.h>

#include "common.cuh"
#include "fcnet_layout.cuh"
#include "fcnet_tc_layout.cuh"

namespace ddrl {

using SgdTail = ddrl_sgd_tail;   // include/ddrl_b200.h; theta == nullptr disables the tail

__device__ __forceinline__ unsigned int ld_acquire_u32(const unsigned int* p) {
    unsigned int v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long ld_relaxed_sys_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_sys_u64(unsigned long long* p, unsigned long long v) {
    asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// one thread, after a __syncthreads(): arrive (gpu-scope RELEASE: cumulative over the CTA's writes ordered before it by
// the barrier — no separate __threadfence) and spin (tight acquire loads, no sleep) until `target` CTAs have arrived;
// false on timeout
__device__ __noinline__ static bool grid_group_barrier(unsigned int* ctr, unsigned int target, bool arrive = true) {
    if (arrive) asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(ctr) : "memory");
#pragma unroll 1
    for (unsigned int i = 0; i < 8000000u; ++i) {
        if (ld_acquire_u32(ctr) >= target) return true;
    }
    return false;
}

// barrier-A arrival on its own (one thread, after the __syncthreads() behind the CTA's last partial-gradient store)
__device__ __forceinline__ void sgd_tail_arrive_a(const ddrl_sgd_tail& t, int p) {
    asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(t.barrier_ws + 4 * p) : "memory");
}

__host__ __device__ inline int sgd_slice_len(int NP, int G) { return (((NP + G - 1) / G) + 3) & ~3; }

// Inlined on purpose (an out-of-line call made the whole kernel 6 us slower: parameter struct copied to a local stack,
// ABI register constraints); kernels keep ONE call site.
// Called by every thread of every CTA after the partial gradient (and stat partial) of this CTA has been written.
// smem: 16 * blockDim.x + 256 bytes of (16-byte aligned) shared memory.  Returns false if a barrier or a peer wait timed out.
//
// A launch may run several consecutive SGD steps ("persistent" kernels, ddrl_sgd_tail.nsteps > 1): TailStep carries the
// per-step state the caller keeps in registers.  Barrier counters count up across the steps of a launch (target =
// G * round) and are re-armed by the ticket of the LAST step; between steps the tail ends with an arrival on barrier C
// (all of this policy's Adam slices written) which the caller awaits with sgd_wait_weights() before reloading weights.
struct TailStep {
    int round;           // 1-based step number inside this launch
    bool last;           // last step of the launch: ticket (step counter, sequence, barrier re-arm) instead of barrier C
    float b1p, b2p;      // beta1^t, beta2^t of THIS step (read from beta_pow at kernel entry, advanced by the caller)
    unsigned int seq;    // exchange sequence number of this step (world > 1): *t.seq at kernel entry + round - 1
    int nsteps;          // steps in this launch (the ticket advances the clocks by it)
    unsigned int epoch;  // barrier_ws[4P+1] at kernel entry: steps executed by earlier launches (tags of the sq words)
};
__device__ __forceinline__ TailStep tail_single_step(const SgdTail& t, int p) {
    TailStep ts;
    ts.round = 1; ts.last = true; ts.nsteps = 1;
    ts.b1p = __ldcg(t.beta_pow + p * 2); ts.b2p = __ldcg(t.beta_pow + p * 2 + 1);
    ts.seq = (t.world > 1) ? *t.seq : 0u;
    ts.epoch = __ldcg(t.barrier_ws + 4 * gridDim.y + 1);
    return ts;
}
// wait until every CTA of policy p has finished the Adam slice of step `round` (one thread per CTA calls this)
__device__ __forceinline__ bool sgd_wait_weights(const SgdTail& t, int p, int G, int round) {
#pragma unroll 1
    for (unsigned int i = 0; i < 4000000u; ++i) {
        if (ld_acquire_u32(t.barrier_ws + 4 * p + 2) >= (unsigned)(G * round)) return true;
    }
    return false;
}

// NX: the last NX of the NP parameters are not FCNet variables (the leg-coupling table of SharedDecentralLegID): clipped and
// stepped like the rest, never mapped into the packed weight images.
template <int NX = 0>
__device__ __forceinline__ bool sgd_step_tail(const SgdTail& t, const TailStep& ts, const float* __restrict__ grad_part,
                                              const double* __restrict__ stat_part, int p, int P, int bx, int G, int NP,
                                              int step, int D, int A, float* smem, long long* dbg = nullptr, int npart = 0,
                                              bool arrived = false) {
    // npart: number of gradient partials per policy at grad_part[p][0..npart) (default: one per CTA = G; a kernel that
    // pre-reduces inside thread-block clusters passes the number of clusters)
    // arrived: the caller has already made thread 0 arrive on barrier A (sgd_tail_arrive_a, right behind the __syncthreads()
    // that completed the partial) — so that loads the caller issues in between (the next step's input prefetch) are not
    // ahead of the release and do not lengthen its drain
    if (npart <= 0) npart = G;
#define TAIL_STAMP(i)                                                                                              \
    do {                                                                                                           \
        if (dbg && threadIdx.x == 0) {                                                                             \
            if (blockIdx.x == 0 && blockIdx.y == 0) dbg[i] = clock64();                                            \
            long long gt_;                                                                                         \
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt_));                                                \
            dbg[64 + 8 * (blockIdx.y * gridDim.x + blockIdx.x) + ((i) - 37)] = gt_;   /* 40..43 -> slots 3..6 */     \
        }                                                                                                          \
    } while (0)
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, nw = nt >> 5;
    const int NPs = (NP + 3) & ~3;
    float4* scr = reinterpret_cast<float4*>(smem);
    float* red = smem + 4 * nt;                 // [64]: warp partials, flags
    const int W = t.world > 1 ? t.world : 1;
    bool ok = true;
    // optimizer state of this thread's element: independent of everything below, so the loads fly behind barrier A
    const int S_pf = sgd_slice_len(NP, G);
    const bool pf = S_pf <= nt;
    const int j_pf = bx * S_pf + tid;
    float m_pf = 0.f, v_pf = 0.f, th_pf = 0.f;
    if (pf && tid < S_pf && j_pf < NP) {
        const int64_t k = (int64_t)p * NP + j_pf;
        m_pf = __ldcg(t.m + k); v_pf = __ldcg(t.v + k); th_pf = __ldcg(t.theta + k);
    }
    __syncthreads();
    if (tid == 0) {
        red[40] = 1.f;
        red[39] = grid_group_barrier(t.barrier_ws + 4 * p, (unsigned)(G * ts.round), !arrived) ? 1.f : 0.f;
    }
    __syncthreads();
    ok = ok && red[39] != 0.f;
    TAIL_STAMP(40);

    // ---- slice reduce over the G partials --------------------------------------------------------------------------
    const int S = sgd_slice_len(NP, G), j0 = bx * S, j1 = min(NPs, j0 + S);
    const int ncol4 = max(0, (j1 - j0) >> 2);
    // t.grad_acc: the partials of the policy were ADDED into one vector at L2 (red.global.add, ping-pong kernel): the slice is
    // read once (and zeroed for the next step) instead of being summed over npart partials
    const bool use_acc = t.grad_acc != nullptr;
    float* acc_p = use_acc ? t.grad_acc + (int64_t)p * NPs + j0 : nullptr;
    const int ngrp = (use_acc || ncol4 >= nt) ? 1 : max(1, min(min(8, npart), nt / max(ncol4, 1)));
    const int cpp = nt / ngrp;                  // float4 columns per pass
    const unsigned int seq = ts.seq;
    const unsigned long long want = (unsigned long long)(seq + 1u) << 32;     // flag half of the LL words of this step
    const int par = (int)(seq & 1u);
    const int64_t xstride = (int64_t)G * S;     // words per (rank, policy) in the exchange buffer
    const int64_t xoff = (((int64_t)par * W + t.rank) * P + p) * xstride + j0;   // this rank's slot, same in every buffer
    float* slice_dst = t.grad + (int64_t)p * NP + j0;
    // common case (slice fits one pass of the CTA, `pf`): thread tid owns element j0 + tid and keeps its reduced gradient
    // in a register from here to the Adam update — no global write -> read round trips inside the tail
    float gval = 0.f;
    for (int c0 = 0; c0 < ncol4; c0 += cpp) {
        const int g = tid / cpp, c = c0 + (tid - g * cpp);
        if (!use_acc && g < ngrp && c < ncol4) {
            const float4* src = reinterpret_cast<const float4*>(grad_part + (int64_t)p * G * NPs + j0) + c;
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
            const int64_t pstride = (int64_t)ngrp * (NPs >> 2);
#pragma unroll 1
            for (int i0 = g; i0 < npart; i0 += 8 * ngrp) {     // 8 independent loads in flight, then the (fixed-order) adds
                float4 v[8];
#pragma unroll
                for (int k = 0; k < 8; ++k)
                    v[k] = (i0 + k * ngrp < npart) ? __ldcg(src + (int64_t)i0 * (NPs >> 2) + k * pstride) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                for (int k = 0; k < 8; ++k) { acc.x += v[k].x; acc.y += v[k].y; acc.z += v[k].z; acc.w += v[k].w; }
            }
            scr[g * cpp + (c - c0)] = acc;
        }
        if (!use_acc) __syncthreads();
        const int nf = 4 * min(cpp, ncol4 - c0);
        for (int fb = 0; fb < nf; fb += nt) {      // every thread runs the same trip count: the shuffle below is warp-wide
            const int f = fb + tid;
            const bool act = f < nf;
            const int col = f >> 2, e = f & 3;
            float s = 0.f;
            const int jj = 4 * c0 + f;           // offset inside the slice
            if (act) {
                if (use_acc) {
                    s = __ldcg(acc_p + jj);
                    acc_p[jj] = 0.f;             // re-armed for the next step (ordered before this CTA's barrier-C arrival / ticket)
                } else {
                    for (int gg = 0; gg < ngrp; ++gg) s += reinterpret_cast<const float*>(&scr[gg * cpp + col])[e];
                }
            }
            if (W > 1) {
                // push to every rank's exchange buffer (own copy included).  Two neighbouring elements travel as ONE 16-byte
                // store {value, flag, value, flag} issued by the even lane (NCCL-LL line: each 8-byte half is self-validating,
                // so the store need not be atomic as a whole) — half the NVLink packets of one store per element.
                const float s_nb = __shfl_down_sync(0xffffffffu, s, 1);      // nf is a multiple of 4: lane pairs stay together
                if (act && j0 + jj < NP && (f & 1) == 0) {
                    const unsigned long long w0 = want | (unsigned long long)__float_as_uint(s);
                    if (j0 + jj + 1 < NP) {
                        const unsigned long long w1 = want | (unsigned long long)__float_as_uint(s_nb);
#pragma unroll 1
                        for (int w = 0; w < W; ++w)
                            asm volatile("st.relaxed.sys.global.v2.u64 [%0], {%1, %2};" ::"l"(t.peer_x[w] + xoff + jj), "l"(w0), "l"(w1)
                                         : "memory");
                    } else {
#pragma unroll 1
                        for (int w = 0; w < W; ++w) st_relaxed_sys_u64(t.peer_x[w] + xoff + jj, w0);
                    }
                }
            } else if (act && j0 + jj < NP) {
                slice_dst[jj] = s;
                gval = s;
            }
        }
        if (!pf) __syncthreads();
    }
    // ---- data parallel: wait for the world's words of this step, add them in rank order -------------------------------
    if (W > 1) {
        const unsigned long long* xl = t.peer_x[t.rank] + ((int64_t)par * W * P + p) * xstride + j0;   // + w * P * xstride
        bool got = true;
        const unsigned int want32 = (unsigned int)(want >> 32);
        for (int jj = tid; jj < S && j0 + jj < NP; jj += nt) {
            // all ranks' words are requested together (one L2 round trip when they have already landed — the common case);
            // only the missing ones are polled again
            unsigned long long wd[DDRL_MAX_RANKS];
            unsigned int pending = (1u << W) - 1u;
#pragma unroll 1
            for (unsigned int it = 0; pending != 0u && it < 2000000u; ++it) {
#pragma unroll
                for (int w = 0; w < DDRL_MAX_RANKS; ++w)
                    if ((pending >> w) & 1u) wd[w] = ld_relaxed_sys_u64(xl + (int64_t)w * P * xstride + jj);
#pragma unroll
                for (int w = 0; w < DDRL_MAX_RANKS; ++w)
                    if (((pending >> w) & 1u) && (unsigned int)(wd[w] >> 32) == want32) pending &= ~(1u << w);
            }
            got = got && pending == 0u;
            float s = 0.f;
#pragma unroll
            for (int w = 0; w < DDRL_MAX_RANKS; ++w)
                if (w < W) s += __uint_as_float((unsigned int)wd[w]);      // rank order: identical bits on every rank
            slice_dst[jj] = s;
            gval = s;
        }
        if (!got) red[40] = 0.f;      // benign race: every writer stores the same value
    }
    if (!pf) __syncthreads();
    TAIL_STAMP(41);
    // ---- ||g||^2 of the slice (fixed order) -> barrier B -> global norm ------------------------------------------------
    float ss = 0.f;
    if (pf) {
        ss = gval * gval;        // gval == 0 for threads without an element
    } else {
        for (int jj = tid; jj < S && j0 + jj < NP; jj += nt) {
            const float s = __ldcg(t.grad + (int64_t)p * NP + j0 + jj);
            ss = fmaf(s, s, ss);
        }
    }
    ss = warp_sum(ss);
    if (lane == 0) red[warp] = ss;
    __syncthreads();
    ok = ok && red[40] != 0.f;
    // "barrier B" without a counter: every CTA publishes {||g_slice||^2, epoch tag} as ONE 64-bit word and polls the G words
    // of its policy until they carry this step's tag — no release drain of unrelated stores, no second read of the sums
    // one word per 128-byte line: the pollers of a policy spread over G lines / L2 slices instead of hammering three
    constexpr int SQ_STRIDE = 16;
    unsigned long long* sq64 = reinterpret_cast<unsigned long long*>(t.sq_ws) + (int64_t)p * G * SQ_STRIDE;
    const unsigned int btag = ts.epoch + (unsigned int)ts.round;
    if (warp == 0) {      // the warp partials are added by a shuffle tree (fixed order; a serial loop of one thread over the
        float s = warp_sum(lane < nw ? red[lane] : 0.f);      // 20 warps was ~0.3 us on the critical path of barrier B)
        if (lane == 0)
            asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(sq64 + (int64_t)bx * SQ_STRIDE),
                         "l"(((unsigned long long)btag << 32) | (unsigned long long)__float_as_uint(s)) : "memory");
    }
    // loss statistics of the step (CTA 0 of the policy; warps 1.. sum one stat each over the G partials, which barrier A made
    // visible).  Done HERE, behind this CTA's norm word: every CTA of the policy waits for the slowest publisher, and with the
    // sums ahead of the publication CTA 0 was that one by ~1 us per step (per-CTA globaltimer stamps).
    if (bx == 0 && warp >= 1 && stat_part && t.step_stats) {
        for (int w = warp - 1; w < DDRL_NSTAT; w += nw - 1) {
            double s = 0.0;
            for (int i = lane; i < G; i += 32) s += __ldcg(stat_part + ((int64_t)p * G + i) * DDRL_NSTAT + w);
            s = warp_sum(s);
            if (lane == 0) t.step_stats[((int64_t)step * P + p) * DDRL_NSTAT + w] = s;
        }
    }
    if (warp == 0) {
        float s = 0.f;
        bool got = true;
        for (int i = lane; i < G; i += 32) {
            unsigned long long w64 = 0ull;
            bool hit = false;
#pragma unroll 1
            for (unsigned int it = 0; it < 8000000u; ++it) {
                asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(w64) : "l"(sq64 + (int64_t)i * SQ_STRIDE) : "memory");
                if ((unsigned int)(w64 >> 32) == btag) { hit = true; break; }
            }
            got = got && hit;
            s += __uint_as_float((unsigned int)w64);
        }
        s = warp_sum(s);
        got = __all_sync(0xffffffffu, got);
        if (lane == 0) {
            const float norm = sqrtf(s);
            red[32] = t.grad_clip > 0.f ? t.grad_clip * fminf(1.f / norm, 1.f / t.grad_clip) : 1.f;
            red[39] = got ? 1.f : 0.f;
            if (bx == 0 && t.gnorm_out) t.gnorm_out[p] = norm;
        }
    }
    __syncthreads();
    ok = ok && red[39] != 0.f;
    TAIL_STAMP(42);
    // ---- clip + TF1 Adam on the slice ---------------------------------------------------------------------------------
    const float scale = red[32];
    const float b1p = ts.b1p, b2p = ts.b2p;
    const float alpha = t.lr * sqrtf(1.f - b2p) / (1.f - b1p);
    for (int jj = tid; jj < S && j0 + jj < NP; jj += nt) {
        const int j = j0 + jj;
        const int64_t k = (int64_t)p * NP + j;
        const float gj = (pf ? gval : __ldcg(t.grad + k)) * scale;
        float mj = pf ? m_pf : t.m[k], vj = pf ? v_pf : t.v[k];
        mj += (gj - mj) * (1.f - t.beta1);
        vj += (gj * gj - vj) * (1.f - t.beta2);
        t.m[k] = mj;
        t.v[k] = vj;
        const float tnew = (pf ? th_pf : t.theta[k]) - (mj * alpha) / (sqrtf(vj) + t.eps);
        t.theta[k] = tnew;
        if (NX > 0 && j >= NP - NX) continue;      // (compile-time: no test in the plain FCNet step)
        if (t.fcnet_img) {
            const FcSmem L = fc_smem(D, A, false);
            const FcOffsets o = fc_offsets(D, A);
            int p0, p1;
            fc_img_pos(L, o, D, A, j, p0, p1);
            float* im = t.fcnet_img + (int64_t)p * L.x;
            im[p0] = tnew;
            if (p1 >= 0) im[p1] = tnew;
        }
        if (t.fcnet_tc_img) {
            const TcImg L = tc_img(D, A);
            const FcOffsets o = fc_offsets(D, A);
            bool f16;
            int p0, p1;
            tc_img_pos(L, o, D, A, j, f16, p0, p1);
            unsigned char* im = reinterpret_cast<unsigned char*>(t.fcnet_tc_img) + (int64_t)p * L.bytes;
            if (f16) {
                const float ws = tnew * 256.f;
                const __half hi = __float2half_rn(ws);
                *reinterpret_cast<__half*>(im + p0) = hi;
                *reinterpret_cast<__half*>(im + p1) = __float2half_rn(ws - __half2float(hi));
            } else {
                *reinterpret_cast<float*>(im + p0) = tnew;
            }
        }
    }
    // ---- end of step: barrier-C arrival (more steps follow in this launch) or the done ticket (last step) -----------------
    __syncthreads();
    TAIL_STAMP(43);
    if (tid == 0) {
        if (!ts.last) {
            asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(t.barrier_ws + 4 * p + 2) : "memory");   // Adam slice visible
        } else {
            __threadfence();
            if (bx == 0) {     // every CTA read beta_pow at kernel entry (before its first barrier-A arrival): safe to advance
                t.beta_pow[p * 2] = ts.b1p * t.beta1;
                t.beta_pow[p * 2 + 1] = ts.b2p * t.beta2;
            }
            const unsigned int total = gridDim.x * gridDim.y;
            if (atomicAdd(t.barrier_ws + 4 * P, 1u) == total - 1) {   // last CTA of the grid: clocks, re-arm
                for (int q = 0; q < P; ++q) {
                    t.barrier_ws[4 * q] = 0u;
                    t.barrier_ws[4 * q + 1] = 0u;
                    t.barrier_ws[4 * q + 2] = 0u;
                }
                t.barrier_ws[4 * P + 1] = ts.epoch + (unsigned int)ts.nsteps;   // every CTA read it at kernel entry
                if (t.step_ctr) *t.step_ctr += ts.nsteps;
                if (t.seq) *t.seq = ts.seq + 1u;
                t.barrier_ws[4 * P] = 0u;
                __threadfence();
            }
        }
        if (!ok && t.status) atomicOr(t.status, 64);
    }
    return ok;
#undef TAIL_STAMP
}

// =====================================================================================================================
// "LL" tail (ping-pong tcgen05 kernel, ddrl_sgd_tail.ll_ws != NULL): the same arithmetic as sgd_step_tail, but the partial
// gradients reach the slice owners as self-validating 64-bit words {fp32 payload, step tag} (NCCL-"LL" style) instead of
// plain data behind a release / acquire barrier:
//
//   write-out   each CTA stores its partial gradient (and its 8 float64 loss statistics as 16 half words) as LL words, then
//               ONE tagged "done" word — relaxed stores, no fence, no drain
//   reduce      the owner of slice bx polls the G done words (one warp), pulls the G slices into shared memory with TMA bulk
//               copies (cp.async.bulk + mbarrier complete_tx: one L2 round trip, no registers) and adds them in a fixed order,
//               checking every word's tag (a word that is not this step's yet -> the copy is repeated)
//   [world > 1] peer exchange, norm exchange ("barrier B"), clip + Adam, barrier-C arrival: as in sgd_step_tail
//
// It removes barrier A (store drain + atomic + poll, ~2 us) and turns the slice reduce into one bulk round trip.  The buffer
// is single: a CTA writes the partial of step s+1 only after it passed barrier C of step s, which every owner reaches
// after it has consumed the partials of step s.  Tags are the global step count (ts.epoch + round >= 1); the workspace
// starts zeroed.  All sums keep a fixed order: bit-reproducible.
__host__ __device__ inline int ll_part_words(int NP) { return ((NP + 3) & ~3) + 2 * DDRL_NSTAT; }
constexpr int LL_FLAG_STRIDE = 16;      // one done word per 128-byte line
__host__ __device__ inline int64_t ll_total_words(int P, int G, int NP) {
    return (int64_t)P * G * ll_part_words(NP) + (int64_t)P * G * LL_FLAG_STRIDE;
}
constexpr int LL_STAGE_BYTES = 88 * 1024;      // shared-memory staging of the slice copies (dead activation buffers)

__device__ __forceinline__ void ll_st1(unsigned long long* p, unsigned int payload, unsigned int tag) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(((unsigned long long)tag << 32) | payload) : "memory");
}
__device__ __forceinline__ void ll_st2(unsigned long long* p, unsigned int a, unsigned int b, unsigned int tag) {
    const unsigned long long t = (unsigned long long)tag << 32;
    asm volatile("st.relaxed.gpu.global.v2.u64 [%0], {%1, %2};" ::"l"(p), "l"(t | a), "l"(t | b) : "memory");
}
__device__ __forceinline__ void ll_ld2(const unsigned long long* p, unsigned long long& a, unsigned long long& b) {
    asm volatile("ld.relaxed.gpu.global.v2.u64 {%0, %1}, [%2];" : "=l"(a), "=l"(b) : "l"(p) : "memory");
}
__device__ __forceinline__ unsigned long long ll_ld1(const unsigned long long* p) {
    unsigned long long a;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(a) : "l"(p) : "memory");
    return a;
}
constexpr unsigned int LL_SPINS = 4000000u;

// TMA bulk copy global -> shared (bytes % 16 == 0, both addresses 16-byte aligned), completion counted on an mbarrier
__device__ __forceinline__ void bulk_g2s(unsigned int smem_dst, const void* gsrc, unsigned int bytes, unsigned int mbar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_dst), "l"(gsrc),
                 "r"(bytes), "r"(mbar)
                 : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned int mbar, unsigned int bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_wait_parity(unsigned int mbar, unsigned int parity) {
#pragma unroll 1
    for (unsigned int i = 0; i < 20000000u; ++i) {
        unsigned int ok;
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.b32 %0, 1, 0, p;\n\t}\n"
                     : "=r"(ok) : "r"(mbar), "r"(parity) : "memory");
        if (ok) return true;
    }
    return false;
}

// Requires sgd_slice_len(NP, G) <= blockDim.x (thread tid owns element bx * S + tid of the slice).
//   smem   16 * blockDim.x + 256 bytes of scratch (16-byte aligned), disjoint from `stage`
//   stage  LL_STAGE_BYTES of shared memory (16-byte aligned) for the slice copies
//   mbar   shared::cta address of an mbarrier initialised with count 1; *mbar_phase = its current parity (kept by the caller)
__device__ __forceinline__ bool sgd_step_tail_ll(const SgdTail& t, const TailStep& ts, int p, int P, int bx, int G, int NP, int step,
                                                 int D, int A, float* smem, unsigned char* stage, unsigned int mbar,
                                                 unsigned int& mbar_phase, long long* dbg = nullptr) {
#define TAIL_STAMP(i)                                                                                              \
    do {                                                                                                           \
        if (dbg && threadIdx.x == 0) {                                                                             \
            if (blockIdx.x == 0 && blockIdx.y == 0) dbg[i] = clock64();                                            \
            long long gt_;                                                                                         \
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt_));                                                \
            dbg[64 + 8 * (blockIdx.y * gridDim.x + blockIdx.x) + ((i) - 37)] = gt_;   /* 40..43 -> slots 3..6 */     \
        }                                                                                                          \
    } while (0)
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, nw = nt >> 5;
    const int NPs = (NP + 3) & ~3, LLW = ll_part_words(NP);
    const unsigned int tag = ts.epoch + (unsigned int)ts.round;
    float* red = smem + 4 * nt;                         // [64]: warp partials, flags
    const int W = t.world > 1 ? t.world : 1;
    bool ok = true;
    const int S = sgd_slice_len(NP, G), j0 = bx * S, j1 = min(NPs, j0 + S), len = max(0, j1 - j0);
    const int j_own = j0 + tid;
    const bool own = tid < S && j_own < NP;
    unsigned long long* flags = t.ll_ws + (int64_t)P * G * LLW + (int64_t)p * G * LL_FLAG_STRIDE;
    // caller: __syncthreads() after the write-out -> every LL store of this CTA has been issued
    if (tid == 0) {
        ll_st1(flags + (int64_t)bx * LL_FLAG_STRIDE, 0u, tag);
        red[40] = 1.f;
        red[41] = 0.f;
    }
    // optimizer state of this thread's element: independent of the reduce, the loads fly behind it
    float m_pf = 0.f, v_pf = 0.f, th_pf = 0.f;
    if (own) {
        const int64_t k = (int64_t)p * NP + j_own;
        m_pf = __ldcg(t.m + k); v_pf = __ldcg(t.v + k); th_pf = __ldcg(t.theta + k);
    }
    // ---- wait for the G done words (warp 0), then pull the slices: chunks of `pc` partials per bulk round ---------------
    const unsigned int slice_bytes = (unsigned int)len * 8u;
    const int pc = slice_bytes > 0 ? min(G, (int)(LL_STAGE_BYTES / slice_bytes)) : G;      // partials per staging round
    if (warp == 0) {
        bool got = true;
        for (int i = lane; i < G; i += 32) {
            bool hit = false;
#pragma unroll 1
            for (unsigned int it = 0; it < 8000000u; ++it) {
                if ((unsigned int)(ll_ld1(flags + (int64_t)i * LL_FLAG_STRIDE) >> 32) == tag) { hit = true; break; }
            }
            got = got && hit;
        }
        got = __all_sync(0xffffffffu, got);
        if (lane == 0 && !got) red[40] = 0.f;
    }
    TAIL_STAMP(40);
    float gsum = 0.f;
    const unsigned long long* stg = reinterpret_cast<const unsigned long long*>(stage);
    const unsigned int stage_s = (unsigned int)__cvta_generic_to_shared(stage);
#pragma unroll 1
    for (int c0 = 0; c0 < G && len > 0; c0 += pc) {
        const int nc = min(pc, G - c0);
#pragma unroll 1
        for (int attempt = 0; attempt < 64; ++attempt) {
            __syncthreads();      // done words seen (first round) / previous use of the staging buffer over
            if (warp == 0) {
                if (lane == 0) mbar_expect_tx(mbar, (unsigned int)nc * slice_bytes);
                __syncwarp();
                for (int i = lane; i < nc; i += 32)
                    bulk_g2s(stage_s + (unsigned int)i * slice_bytes, t.ll_ws + ((int64_t)p * G + c0 + i) * LLW + j0, slice_bytes, mbar);
            }
            if (!mbar_wait_parity(mbar, mbar_phase)) ok = false;
            mbar_phase ^= 1u;
            float part = 0.f;
            bool bad = false;
            if (tid < len) {
#pragma unroll 4
                for (int i = 0; i < nc; ++i) {
                    const unsigned long long w = stg[(int64_t)i * len + tid];
                    bad = bad || (unsigned int)(w >> 32) != tag;
                    part += __uint_as_float((unsigned int)w);
                }
            }
            if (!__syncthreads_or(bad ? 1 : 0)) { gsum += part; break; }      // all words were this step's: partial order fixed
            if (attempt == 63) ok = false;
        }
    }
    float gval = 0.f;      // this thread's reduced gradient element (register-resident up to the Adam update)
    {
        const float s = gsum;
        const bool act = tid < len;
        const int64_t xstride = (int64_t)G * S;
        float* slice_dst = t.grad + (int64_t)p * NP + j0;
        if (W > 1) {
            // push to every rank's exchange buffer (own copy included), two neighbouring elements as ONE 16-byte store
            const unsigned int seq = ts.seq;
            const unsigned long long want = (unsigned long long)(seq + 1u) << 32;
            const int par = (int)(seq & 1u);
            const int64_t xoff = (((int64_t)par * W + t.rank) * P + p) * xstride + j0;
            const float s_nb = __shfl_down_sync(0xffffffffu, s, 1);      // len is even: pairs never straddle a warp edge
            if (act && j_own < NP && (tid & 1) == 0) {
                const unsigned long long w0 = want | (unsigned long long)__float_as_uint(s);
                if (j_own + 1 < NP) {
                    const unsigned long long w1 = want | (unsigned long long)__float_as_uint(s_nb);
#pragma unroll 1
                    for (int w = 0; w < W; ++w)
                        asm volatile("st.relaxed.sys.global.v2.u64 [%0], {%1, %2};" ::"l"(t.peer_x[w] + xoff + tid), "l"(w0), "l"(w1)
                                     : "memory");
                } else {
#pragma unroll 1
                    for (int w = 0; w < W; ++w) st_relaxed_sys_u64(t.peer_x[w] + xoff + tid, w0);
                }
            }
            // wait for the world's words of this step, add them in rank order
            if (own) {
                const unsigned long long* xl = t.peer_x[t.rank] + ((int64_t)par * W * P + p) * xstride + j0 + tid;
                const unsigned int want32 = seq + 1u;
                unsigned long long wd[DDRL_MAX_RANKS];
                unsigned int pending = (1u << W) - 1u;
#pragma unroll 1
                for (unsigned int it = 0; pending != 0u && it < 2000000u; ++it) {
#pragma unroll
                    for (int w = 0; w < DDRL_MAX_RANKS; ++w)
                        if ((pending >> w) & 1u) wd[w] = ld_relaxed_sys_u64(xl + (int64_t)w * P * xstride);
#pragma unroll
                    for (int w = 0; w < DDRL_MAX_RANKS; ++w)
                        if (((pending >> w) & 1u) && (unsigned int)(wd[w] >> 32) == want32) pending &= ~(1u << w);
                }
                ok = ok && pending == 0u;
                float sw = 0.f;
#pragma unroll
                for (int w = 0; w < DDRL_MAX_RANKS; ++w)
                    if (w < W) sw += __uint_as_float((unsigned int)wd[w]);      // rank order: identical bits on every rank
                slice_dst[tid] = sw;
                gval = sw;
            }
        } else if (own) {
            slice_dst[tid] = s;
            gval = s;
        }
    }
    // loss statistics: CTA 0 of the policy, warp w sums stat w over the G partials (two 32-bit halves per float64)
    if (bx == 0 && warp < DDRL_NSTAT && t.step_stats) {
        double s = 0.0;
        bool got = true;
        for (int i = lane; i < G; i += 32) {
            const unsigned long long* src = t.ll_ws + ((int64_t)p * G + i) * LLW + NPs + 2 * warp;
            unsigned long long a = 0ull, b = 0ull;
            bool hit = false;
#pragma unroll 1
            for (unsigned int it = 0; it < LL_SPINS; ++it) {
                ll_ld2(src, a, b);
                if ((unsigned int)(a >> 32) == tag && (unsigned int)(b >> 32) == tag) { hit = true; break; }
            }
            got = got && hit;
            s += __longlong_as_double((long long)(((b & 0xffffffffull) << 32) | (a & 0xffffffffull)));
        }
        s = warp_sum(s);
        ok = ok && got;
        if (lane == 0) t.step_stats[((int64_t)step * P + p) * DDRL_NSTAT + warp] = s;
    }
    TAIL_STAMP(41);
    // ---- ||g||^2 of the slice (fixed order) -> tagged words ("barrier B") -> global norm -------------------------------
    float ss = warp_sum(gval * gval);
    if (lane == 0) red[warp] = ss;
    if (!ok) red[40] = 0.f;      // benign race: every writer stores the same value
    __syncthreads();
    constexpr int SQ_STRIDE = 16;
    unsigned long long* sq64 = reinterpret_cast<unsigned long long*>(t.sq_ws) + (int64_t)p * G * SQ_STRIDE;
    if (tid == 0) {
        float s = 0.f;
        for (int w = 0; w < nw; ++w) s += red[w];
        asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(sq64 + (int64_t)bx * SQ_STRIDE),
                     "l"(((unsigned long long)tag << 32) | (unsigned long long)__float_as_uint(s)) : "memory");
    }
    if (warp == 0) {
        float s = 0.f;
        bool got = true;
        for (int i = lane; i < G; i += 32) {
            unsigned long long w64 = 0ull;
            bool hit = false;
#pragma unroll 1
            for (unsigned int it = 0; it < 8000000u; ++it) {
                w64 = ll_ld1(sq64 + (int64_t)i * SQ_STRIDE);
                if ((unsigned int)(w64 >> 32) == tag) { hit = true; break; }
            }
            got = got && hit;
            s += __uint_as_float((unsigned int)w64);
        }
        s = warp_sum(s);
        got = __all_sync(0xffffffffu, got);
        if (lane == 0) {
            const float norm = sqrtf(s);
            red[32] = t.grad_clip > 0.f ? t.grad_clip * fminf(1.f / norm, 1.f / t.grad_clip) : 1.f;
            red[39] = got ? 1.f : 0.f;
            if (bx == 0 && t.gnorm_out) t.gnorm_out[p] = norm;
        }
    }
    __syncthreads();
    ok = red[39] != 0.f && red[40] != 0.f;
    TAIL_STAMP(42);
    // ---- clip + TF1 Adam on the slice; the tensor-core image first (it is what barrier C publishes) ----------------------
    if (own) {
        const float scale = red[32];
        const float alpha = t.lr * sqrtf(1.f - ts.b2p) / (1.f - ts.b1p);
        const int64_t k = (int64_t)p * NP + j_own;
        const float gj = gval * scale;
        float mj = m_pf, vj = v_pf;
        mj += (gj - mj) * (1.f - t.beta1);
        vj += (gj * gj - vj) * (1.f - t.beta2);
        const float tnew = th_pf - (mj * alpha) / (sqrtf(vj) + t.eps);
        const TcImg L = tc_img(D, A);
        const FcOffsets o = fc_offsets(D, A);
        bool f16;
        int p0, p1;
        tc_img_pos(L, o, D, A, j_own, f16, p0, p1);
        unsigned char* im = reinterpret_cast<unsigned char*>(t.fcnet_tc_img) + (int64_t)p * L.bytes;
        if (f16) {
            const float ws = tnew * 256.f;
            const __half hi = __float2half_rn(ws);
            *reinterpret_cast<__half*>(im + p0) = hi;
            *reinterpret_cast<__half*>(im + p1) = __float2half_rn(ws - __half2float(hi));
        } else {
            *reinterpret_cast<float*>(im + p0) = tnew;
        }
        t.m[k] = mj;
        t.v[k] = vj;
        t.theta[k] = tnew;
    }
    // ---- end of step: barrier-C arrival (more steps follow in this launch) or the done ticket (last step) -----------------
    __syncthreads();
    TAIL_STAMP(43);
    if (tid == 0) {
        if (!ts.last) {
            asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(t.barrier_ws + 4 * p + 2) : "memory");   // Adam slice visible
        } else {
            __threadfence();
            if (bx == 0) {     // every CTA read beta_pow at kernel entry: safe to advance
                t.beta_pow[p * 2] = ts.b1p * t.beta1;
                t.beta_pow[p * 2 + 1] = ts.b2p * t.beta2;
            }
            const unsigned int total = gridDim.x * gridDim.y;
            if (atomicAdd(t.barrier_ws + 4 * P, 1u) == total - 1) {   // last CTA of the grid: clocks, re-arm
                for (int q = 0; q < P; ++q) {
                    t.barrier_ws[4 * q] = 0u;
                    t.barrier_ws[4 * q + 1] = 0u;
                    t.barrier_ws[4 * q + 2] = 0u;
                }
                t.barrier_ws[4 * P + 1] = ts.epoch + (unsigned int)ts.nsteps;   // every CTA read it at kernel entry
                if (t.step_ctr) *t.step_ctr += ts.nsteps;
                if (t.seq) *t.seq = ts.seq + 1u;
                t.barrier_ws[4 * P] = 0u;
                __threadfence();
            }
        }
        if (!ok && t.status) atomicOr(t.status, 64);
    }
    return ok;
#undef TAIL_STAMP
}

// Host-side validation shared by the launchers.
inline int sgd_tail_check(const ddrl_sgd_tail* tail, int ctas_total, const char* who) {
    DDRL_REQUIRE(tail->theta && tail->m && tail->v && tail->beta_pow && tail->grad && tail->barrier_ws && tail->sq_ws,
                 DDRL_E_BADARG, "%s: incomplete fused tail", who);
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    DDRL_REQUIRE(ctas_total <= sms, DDRL_E_BADARG, "%s: fused tail needs all %d CTAs co-resident (%d SMs)", who, ctas_total, sms);
    DDRL_REQUIRE(tail->nsteps >= 0, DDRL_E_BADARG, "%s: fused tail: nsteps must be >= 0", who);
    DDRL_REQUIRE(!tail->ll_ws || tail->fcnet_tc_img, DDRL_E_BADARG, "%s: fused tail: ll_ws needs the tensor-core image", who);
    if (tail->world > 1) {
        DDRL_REQUIRE(tail->world <= DDRL_MAX_RANKS && tail->rank >= 0 && tail->rank < tail->world && tail->seq, DDRL_E_BADARG,
                     "%s: fused tail: bad world/rank/seq (world <= %d)", who, DDRL_MAX_RANKS);
        for (int w = 0; w < tail->world; ++w)
            DDRL_REQUIRE(tail->peer_x[w], DDRL_E_BADARG, "%s: fused tail: peer buffer %d missing", who, w);
    }
    return DDRL_OK;
}

// The tail descriptor one launch receives (SgdTail{}: no fused tail).  Only a kernel that ADDS its partial gradient into
// the accumulation vector keeps grad_acc: the ping-pong tcgen05 step without thread-block clusters and without the LL tail
// (`pingpong_unclustered`).  Every other kernel writes per-CTA partials, which the tail must then read.
inline SgdTail launch_tail(const ddrl_sgd_tail* tail, bool pingpong_unclustered) {
    SgdTail t = tail ? *tail : SgdTail{};
    if (!pingpong_unclustered || t.ll_ws) t.grad_acc = nullptr;
    return t;
}

}  // namespace ddrl

// GraphNet (models/graph_net.py:10-45): hyper-network leg encoder -> MPNN over the 4-leg graph ->
// gather controlled node -> linear head; wrapper with separate actor and critic nets
// (models/shared_graphnet_glorot_uniform_init.py:21-58).  Also the GCN layer (models/gcn.py:7-37).
//
// One CTA of 256 threads keeps ONE net's weights on chip for its whole life and walks over rows:
//   thread (h = tid/4, fs = tid%4) owns the encoder columns j = f*64 + h for f = fs, fs+4, ... (<19):
//     w_j = tanh(e . Wenc[:, j] + b_j)   (e = state[n][19:23]),  x[n][h] = tanh(sum_f state[n][f] w_j)
//     -> the sum over f is 5 local terms + two shuffles, no block barrier;
//   only the nodes the output depends on are encoded: the controlled node and its in-neighbours
//     (adj[s][idx] != 0), i.e. 3 of 4 on the ring — identical result, 25 % less work;
//   MPNN: y[h'] = tanh(sum_h x_i[h] Wupd[h][h'] + mean_s(x_s)[h] Wmsg[h][h']); thread (h' = tid/4,
//     part = tid%4) owns h = 4i + part of both matrices in registers (mean before the transform is the
//     same linear map as the reference's per-edge transform + segment mean);
//   backward mirrors it with the transposed use of Wupd/Wmsg served from shared memory (stride 68 =>
//     conflict free) and per-thread gradient accumulators in registers; per-CTA partials leave once.
#include <math.h>
#include <stdlib.h>

#include <algorithm>

#include "common.cuh"
#include "ppo_loss.cuh"

namespace ddrl {

// tanh = sign(x) * (1 - 2 / (exp(2|x|) + 1)) on the MUFU pipe (ex2 + rcp): absolute error <= 2.4e-7 over the whole range
// (tanhf: 1.2e-7) at a third of the instructions — the hyper-network evaluates 1216 tanh per node.
__device__ __forceinline__ float gn_tanh(float x) {
    float t, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(fabsf(x) * 2.885390081777927f));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(t + 1.f));
    return copysignf(fmaf(-2.f, r, 1.f), x);
}

constexpr int GH = DDRL_HIDDEN;          // 64
constexpr int GF = DDRL_GN_FEATS;        // 19
constexpr int GE = DDRL_GN_ENC_IN;       // 4
constexpr int GS = GF + GE;              // 23 floats per node
constexpr int GN = DDRL_GN_NODES;        // 4
constexpr int GT2 = 256;
constexpr int GK = 5;                    // encoder columns per thread
constexpr int GLD = 68;                  // smem stride of Wupd/Wmsg for the transposed use
constexpr int GMAXO = 2 * DDRL_MAX_ACT;  // 16
constexpr int GIN = GN * GS + GN * GN + 1 + GMAXO;  // staged floats per row: state, adj, idx, dout

struct GnOffsets { int We, be, Wm, Wu, Wo, bo, NP; };
__host__ __device__ inline GnOffsets gn_offsets(int O) {
    GnOffsets o;
    int p = 0;
    o.We = p; p += GE * GF * GH;
    o.be = p; p += GF * GH;
    o.Wm = p; p += GH * GH;
    o.Wu = p; p += GH * GH;
    o.Wo = p; p += GH * O;
    o.bo = p; p += O;
    o.NP = p;
    return o;
}

struct GnRow {      // per-row graph structure, identical in all threads; slot == node id (static indexing)
    int idx, cnt;
    bool need[GN];      // node must be encoded (controlled node or one of its in-neighbours)
    bool is_snd[GN];    // node sends to idx
};

__device__ __forceinline__ GnRow gn_row(const float* sin) {
    GnRow g;
    g.idx = min(max(__float_as_int(sin[GN * GS + GN * GN]), 0), GN - 1);
    g.cnt = 0;
#pragma unroll
    for (int n = 0; n < GN; ++n) {
        const bool snd = sin[GN * GS + n * GN + g.idx] != 0.f;
        g.is_snd[n] = snd;
        g.need[n] = snd || n == g.idx;
        g.cnt += snd ? 1 : 0;
    }
    return g;
}

template <bool BWD>
__global__ void __launch_bounds__(GT2, 1)
graphnet_kernel(const float* __restrict__ theta, const int32_t* __restrict__ node_idx, const float* __restrict__ state,
                const float* __restrict__ adj, const float* __restrict__ dlogits, const float* __restrict__ dvalue,
                int64_t B, int A, float* __restrict__ logits, float* __restrict__ value, float* __restrict__ grad_part) {
    __shared__ __align__(16) float sIn[2][GIN + 3];
    __shared__ float sX[GN][GH];
    __shared__ float sD[GH];
    __shared__ float sOut[GT2 / 32][GMAXO];
    __shared__ __align__(16) float sWuT[BWD ? GH * GLD : 1];
    __shared__ __align__(16) float sWmT[BWD ? GH * GLD : 1];

    const int net = blockIdx.y;                 // 0 actor, 1 critic
    const int O = net == 0 ? 2 * A : 1;
    const GnOffsets oa = gn_offsets(2 * A);
    const GnOffsets o = gn_offsets(O);
    const int net_base = net == 0 ? 0 : oa.NP;
    const float* th = theta + net_base;
    const int tid = threadIdx.x, h = tid >> 2, fs = tid & 3, lane = tid & 31, warp = tid >> 5;
    const int G = gridDim.x, bx = blockIdx.x;

    // ---- weights -> registers / shared --------------------------------------------------------------
    float We[GK][GE], be[GK];
#pragma unroll
    for (int k = 0; k < GK; ++k) {
        const int f = fs + 4 * k;
        const bool ok = f < GF;
#pragma unroll
        for (int q = 0; q < GE; ++q) We[k][q] = ok ? th[o.We + q * GF * GH + f * GH + h] : 0.f;
        be[k] = ok ? th[o.be + f * GH + h] : 0.f;
    }
    float Wu[16], Wm[16];   // forward use: thread (h' = h, part = fs) owns input rows 4i + part
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        Wu[i] = th[o.Wu + (4 * i + fs) * GH + h];
        Wm[i] = th[o.Wm + (4 * i + fs) * GH + h];
    }
    float Wo[GMAXO];
#pragma unroll
    for (int q = 0; q < GMAXO; ++q) Wo[q] = q < O ? th[o.Wo + h * O + q] : 0.f;
    if (BWD) {
        for (int i = tid; i < GH * GH; i += GT2) {
            const int r = i >> 6, c = i & 63;
            sWuT[r * GLD + c] = th[o.Wu + i];
            sWmT[r * GLD + c] = th[o.Wm + i];
        }
    }
    float gWe[GK][GE], gbe[GK], gWu[16], gWm[16], gWo[GMAXO], gbo = 0.f;
    if (BWD) {
#pragma unroll
        for (int k = 0; k < GK; ++k) {
            gbe[k] = 0.f;
#pragma unroll
            for (int q = 0; q < GE; ++q) gWe[k][q] = 0.f;
        }
#pragma unroll
        for (int i = 0; i < 16; ++i) { gWu[i] = 0.f; gWm[i] = 0.f; }
#pragma unroll
        for (int q = 0; q < GMAXO; ++q) gWo[q] = 0.f;
    }

    // ---- row staging: state[92] adj[16] idx[1] dout[O] ------------------------------------------------
    auto fetch = [&](int64_t b) -> float {
        if (b >= B) return 0.f;
        if (tid < GN * GS) return state[b * GN * GS + tid];
        if (tid < GN * GS + GN * GN) return adj[b * GN * GN + (tid - GN * GS)];
        if (tid == GN * GS + GN * GN) return __int_as_float(node_idx[b]);
        if (BWD) {
            const int q = tid - (GN * GS + GN * GN + 1);
            if (q < O) return net == 0 ? dlogits[b * O + q] : dvalue[b];
        }
        return 0.f;
    };
    int cur = 0;
    if (tid < GIN) sIn[0][tid] = fetch(bx);
    __syncthreads();

    for (int64_t b = bx; b < B; b += G) {
        const float* sin = sIn[cur];
        const float pre_next = tid < GIN ? fetch(b + G) : 0.f;   // prefetch the next row (registers)
        const GnRow g = gn_row(sin);

        // ---- encoder for the needed nodes ---------------------------------------------------------
        float wk[GN][GK], xk[GN];
#pragma unroll
        for (int i = 0; i < GN; ++i) {
            xk[i] = 0.f;
            if (g.need[i]) {
                const float* st = sin + i * GS;
                const float e0 = st[GF], e1 = st[GF + 1], e2 = st[GF + 2], e3 = st[GF + 3];
                float part = 0.f;
#pragma unroll
                for (int k = 0; k < GK; ++k) {
                    const int f = fs + 4 * k;
                    float pre = be[k];
                    pre = fmaf(e0, We[k][0], pre);
                    pre = fmaf(e1, We[k][1], pre);
                    pre = fmaf(e2, We[k][2], pre);
                    pre = fmaf(e3, We[k][3], pre);
                    const float w = gn_tanh(pre);
                    wk[i][k] = w;
                    if (f < GF) part = fmaf(st[f], w, part);
                }
                part += __shfl_xor_sync(0xffffffffu, part, 1);
                part += __shfl_xor_sync(0xffffffffu, part, 2);
                xk[i] = gn_tanh(part);
                if (fs == 0) sX[i][h] = xk[i];
            }
        }
        __syncthreads();   // S1: x of all needed nodes visible

        // ---- MPNN for the controlled node: thread (h' = h, part = fs) ---------------------------------
        const float inv_cnt = g.cnt > 0 ? 1.f / (float)g.cnt : 0.f;
        float pre = 0.f;
        float xi[16], xm[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const int hh = 4 * i + fs;
            xi[i] = sX[g.idx][hh];
            float s = 0.f;
#pragma unroll
            for (int n = 0; n < GN; ++n)
                if (g.is_snd[n]) s += sX[n][hh];
            xm[i] = s * inv_cnt;
            pre = fmaf(xi[i], Wu[i], pre);
            pre = fmaf(xm[i], Wm[i], pre);
        }
        pre += __shfl_xor_sync(0xffffffffu, pre, 1);
        pre += __shfl_xor_sync(0xffffffffu, pre, 2);
        const float y = gn_tanh(pre);

        if (!BWD) {
            // head: out[q] = sum_h' y[h'] Wout[h'][q] + b[q]; warp shuffle over the 8 h' of the warp, then 8 warps
#pragma unroll
            for (int q = 0; q < GMAXO; ++q) {
                if (q < O) {
                    float v = fs == 0 ? y * Wo[q] : 0.f;
#pragma unroll
                    for (int s = 16; s > 0; s >>= 1) v += __shfl_xor_sync(0xffffffffu, v, s);
                    if (lane == 0) sOut[warp][q] = v;
                }
            }
            if (tid < GIN) sIn[cur ^ 1][tid] = pre_next;
            __syncthreads();   // S2
            if (tid < O) {
                float v = th[o.bo + tid];
#pragma unroll
                for (int w = 0; w < GT2 / 32; ++w) v += sOut[w][tid];
                if (net == 0) logits[b * O + tid] = v; else value[b] = v;
            }
        } else {
            const float* dout = sin + GN * GS + GN * GN + 1;
            float dy = 0.f;
#pragma unroll
            for (int q = 0; q < GMAXO; ++q)
                if (q < O) {
                    dy = fmaf(dout[q], Wo[q], dy);
                    gWo[q] = fmaf(y, dout[q], gWo[q]);
                }
            if (tid < O) gbo += dout[tid];
            const float dpre = dy * (1.f - y * y);
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                gWu[i] = fmaf(xi[i], dpre, gWu[i]);
                gWm[i] = fmaf(xm[i], dpre, gWm[i]);
            }
            if (fs == 0) sD[h] = dpre;
            if (tid < GIN) sIn[cur ^ 1][tid] = pre_next;
            __syncthreads();   // S2: dpre visible
            // dx_i[h], dxm[h]: thread (h, fs) sums over h' = 4i + fs with the transposed use from shared memory
            float dxi = 0.f, dxm = 0.f;
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const float d = sD[4 * i + fs];
                dxi = fmaf(sWuT[h * GLD + 4 * i + fs], d, dxi);
                dxm = fmaf(sWmT[h * GLD + 4 * i + fs], d, dxm);
            }
            dxi += __shfl_xor_sync(0xffffffffu, dxi, 1);
            dxi += __shfl_xor_sync(0xffffffffu, dxi, 2);
            dxm += __shfl_xor_sync(0xffffffffu, dxm, 1);
            dxm += __shfl_xor_sync(0xffffffffu, dxm, 2);
            dxm *= inv_cnt;
#pragma unroll
            for (int i = 0; i < GN; ++i) {
                if (g.need[i]) {
                    const float dx = (i == g.idx ? dxi : 0.f) + (g.is_snd[i] ? dxm : 0.f);
                    const float dpx = dx * (1.f - xk[i] * xk[i]);
                    const float* st = sin + i * GS;
                    const float e0 = st[GF], e1 = st[GF + 1], e2 = st[GF + 2], e3 = st[GF + 3];
#pragma unroll
                    for (int k = 0; k < GK; ++k) {
                        const int f = fs + 4 * k;
                        if (f < GF) {
                            const float w = wk[i][k];
                            const float dpw = dpx * st[f] * (1.f - w * w);
                            gWe[k][0] = fmaf(e0, dpw, gWe[k][0]);
                            gWe[k][1] = fmaf(e1, dpw, gWe[k][1]);
                            gWe[k][2] = fmaf(e2, dpw, gWe[k][2]);
                            gWe[k][3] = fmaf(e3, dpw, gWe[k][3]);
                            gbe[k] += dpw;
                        }
                    }
                }
            }
        }
        cur ^= 1;
    }

    if (BWD) {
        float* gp = grad_part + (int64_t)bx * ((oa.NP + gn_offsets(1).NP + 3) & ~3) + net_base;
#pragma unroll
        for (int k = 0; k < GK; ++k) {
            const int f = fs + 4 * k;
            if (f < GF) {
#pragma unroll
                for (int q = 0; q < GE; ++q) gp[o.We + q * GF * GH + f * GH + h] = gWe[k][q];
                gp[o.be + f * GH + h] = gbe[k];
            }
        }
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            gp[o.Wu + (4 * i + fs) * GH + h] = gWu[i];
            gp[o.Wm + (4 * i + fs) * GH + h] = gWm[i];
        }
        if (fs == 0)
#pragma unroll
            for (int q = 0; q < GMAXO; ++q)
                if (q < O) gp[o.Wo + h * O + q] = gWo[q];
        if (tid < O) gp[o.bo + tid] = gbo;
    }
}

// ---- forward only, ONE WARP PER ROW ------------------------------------------------------------------------------------
// The row-per-CTA kernel above pays two block barriers and a cross-warp reduction per row (~1.9 us per row: 426 us for a
// 16 384-row minibatch, profiles/r01_launches_graphnet_summary.csv).  Inference and the SGD-step forward need no gradient
// accumulators, so here one net's weights live in SHARED memory (73 KB, 3 CTAs per SM) and every warp walks over its own
// rows without any block barrier: lane l owns the hidden units l and l + 32,
//   encoder  x[n][h] = tanh(sum_f state[n][f] * tanh(b[f][h] + e . We[:, f, h]))     (conflict-free rows of We / be)
//   MPNN     y[h']   = tanh(sum_h x_idx[h] Wu[h][h'] + mean_s x_s[h] Wm[h][h'])       (x through 1 KB of per-warp smem)
//   head     out[q]  = sum_h' y[h'] Wo[h'][q] + bo[q]                                 (warp shuffle reduction)
// Same arithmetic as graphnet_kernel<false> up to the FP32 summation order.
constexpr int GWF_NT = 256;                   // 8 warps
constexpr int GWF_WARPS = GWF_NT / 32;
constexpr int GWF_ROW = 128;                  // staged floats per row (92 state + 16 adj + idx, padded)
constexpr int GWF_WO = GMAXO + 1;             // stride of the head matrix: lanes hit distinct banks
constexpr int GWF_SMEM_FLOATS = GE * GF * GH + GF * GH + 2 * GH * GH + GH * GWF_WO + GMAXO + GWF_WARPS * GWF_ROW +
                                GWF_WARPS * GN * GH;

// SAMPLE (ddrl_graphnet_act): the actor warps also draw the row's DiagGaussian action from eps [B][A] -> action [B][A],
// logp [B] with dg_sample_kernel's row body (bit-identical to ddrl_dg_sample on the logits written here).
template <bool SAMPLE>
__global__ void __launch_bounds__(GWF_NT, 3)
graphnet_fwd_warp_kernel(const float* __restrict__ theta, const int32_t* __restrict__ node_idx,
                         const float* __restrict__ state, const float* __restrict__ adj, int64_t B, int A,
                         float* __restrict__ logits, float* __restrict__ value, const float* __restrict__ eps,
                         float* __restrict__ action, float* __restrict__ logp) {
    extern __shared__ __align__(16) float gsm[];
    float* sWe = gsm;                           // [GE][GF*GH]
    float* sbe = sWe + GE * GF * GH;            // [GF*GH]
    float* sWu = sbe + GF * GH;                 // [GH][GH]  (input h, output h')
    float* sWm = sWu + GH * GH;
    float* sWo = sWm + GH * GH;                 // [GH][GWF_WO]
    float* sbo = sWo + GH * GWF_WO;             // [GMAXO]
    float* sRowAll = sbo + GMAXO;               // [warps][GWF_ROW]
    float* sXAll = sRowAll + GWF_WARPS * GWF_ROW;   // [warps][GN][GH]

    const int net = blockIdx.y;                 // 0 actor, 1 critic
    const int O = net == 0 ? 2 * A : 1;
    const GnOffsets o = gn_offsets(O);
    const float* th = theta + (net == 0 ? 0 : gn_offsets(2 * A).NP);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    for (int i = tid; i < GE * GF * GH; i += GWF_NT) sWe[i] = th[o.We + i];
    for (int i = tid; i < GF * GH; i += GWF_NT) sbe[i] = th[o.be + i];
    for (int i = tid; i < GH * GH; i += GWF_NT) {
        sWu[i] = th[o.Wu + i];
        sWm[i] = th[o.Wm + i];
    }
    for (int i = tid; i < GH * GMAXO; i += GWF_NT) {
        const int hh = i / GMAXO, q = i - hh * GMAXO;
        sWo[hh * GWF_WO + q] = q < O ? th[o.Wo + hh * O + q] : 0.f;
    }
    if (tid < GMAXO) sbo[tid] = tid < O ? th[o.bo + tid] : 0.f;
    __syncthreads();

    float* sRow = sRowAll + warp * GWF_ROW;
    float* sX = sXAll + warp * GN * GH;
    const int64_t stride = (int64_t)gridDim.x * GWF_WARPS;
    for (int64_t b = (int64_t)blockIdx.x * GWF_WARPS + warp; b < B; b += stride) {
        for (int i = lane; i < GN * GS; i += 32) sRow[i] = state[b * GN * GS + i];
        if (lane < GN * GN) sRow[GN * GS + lane] = adj[b * GN * GN + lane];
        if (lane == GN * GN) sRow[GN * GS + GN * GN] = __int_as_float(node_idx[b]);
        __syncwarp();
        const GnRow g = gn_row(sRow);

        // ---- encoder of the needed nodes (controlled node + its in-neighbours): every encoder weight is read from shared
        //      memory ONCE per row and used for all of the row's nodes -----------------------------------------------------
        float e[GN][GE], a0[GN], a1[GN];
#pragma unroll
        for (int n = 0; n < GN; ++n) {
            a0[n] = 0.f;
            a1[n] = 0.f;
#pragma unroll
            for (int q = 0; q < GE; ++q) e[n][q] = sRow[n * GS + GF + q];
        }
#pragma unroll
        for (int f = 0; f < GF; ++f) {
            const int j = f * GH + lane;
            const float b0 = sbe[j], b1 = sbe[j + 32];
            const float w00 = sWe[j], w01 = sWe[j + 32];
            const float w10 = sWe[GF * GH + j], w11 = sWe[GF * GH + j + 32];
            const float w20 = sWe[2 * GF * GH + j], w21 = sWe[2 * GF * GH + j + 32];
            const float w30 = sWe[3 * GF * GH + j], w31 = sWe[3 * GF * GH + j + 32];
#pragma unroll
            for (int n = 0; n < GN; ++n) {
                if (g.need[n]) {                // warp-uniform
                    float p0 = b0, p1 = b1;
                    p0 = fmaf(e[n][0], w00, p0);
                    p1 = fmaf(e[n][0], w01, p1);
                    p0 = fmaf(e[n][1], w10, p0);
                    p1 = fmaf(e[n][1], w11, p1);
                    p0 = fmaf(e[n][2], w20, p0);
                    p1 = fmaf(e[n][2], w21, p1);
                    p0 = fmaf(e[n][3], w30, p0);
                    p1 = fmaf(e[n][3], w31, p1);
                    const float sf = sRow[n * GS + f];
                    a0[n] = fmaf(sf, gn_tanh(p0), a0[n]);
                    a1[n] = fmaf(sf, gn_tanh(p1), a1[n]);
                }
            }
        }
#pragma unroll
        for (int n = 0; n < GN; ++n) {
            if (g.need[n]) {
                sX[n * GH + lane] = gn_tanh(a0[n]);
                sX[n * GH + lane + 32] = gn_tanh(a1[n]);
            }
        }
        __syncwarp();      // x of all needed nodes visible; the staged state is no longer needed

        // ---- MPNN for the controlled node: mean of the senders once per row (into the free staging buffer) ----------------
        const float inv_cnt = g.cnt > 0 ? 1.f / (float)g.cnt : 0.f;
        {
            float m0 = 0.f, m1 = 0.f;
#pragma unroll
            for (int n = 0; n < GN; ++n)
                if (g.is_snd[n]) {
                    m0 += sX[n * GH + lane];
                    m1 += sX[n * GH + lane + 32];
                }
            sRow[lane] = m0 * inv_cnt;
            sRow[lane + 32] = m1 * inv_cnt;
        }
        __syncwarp();
        const float* xs = sX + g.idx * GH;
        float y0 = 0.f, y1 = 0.f;
#pragma unroll 8
        for (int hh = 0; hh < GH; ++hh) {
            const float xi = xs[hh];
            const float xm = sRow[hh];
            y0 = fmaf(xi, sWu[hh * GH + lane], y0);
            y1 = fmaf(xi, sWu[hh * GH + lane + 32], y1);
            y0 = fmaf(xm, sWm[hh * GH + lane], y0);
            y1 = fmaf(xm, sWm[hh * GH + lane + 32], y1);
        }
        y0 = gn_tanh(y0);
        y1 = gn_tanh(y1);

        // ---- head ---------------------------------------------------------------------------------------------------
#pragma unroll
        for (int q = 0; q < GMAXO; ++q) {
            if (q < O) {
                float v = fmaf(y0, sWo[lane * GWF_WO + q], y1 * sWo[(lane + 32) * GWF_WO + q]);
#pragma unroll
                for (int sft = 16; sft > 0; sft >>= 1) v += __shfl_xor_sync(0xffffffffu, v, sft);
                if (lane == q) {
                    v += sbo[q];
                    if (net == 0) logits[b * O + q] = v; else value[b] = v;
                    if (SAMPLE) sRow[GH + q] = v;   // sRow[GH..) is free since the encoder's barrier (the MPNN uses [0, GH))
                }
            }
        }
        if (SAMPLE && net == 0) {
            __syncwarp();
            if (lane == 0) logp[b] = dg_sample_row(sRow + GH, eps + b * A, 0, A, action + b * A);
        }
        __syncwarp();      // every lane is done with sRow / sX before the next row overwrites them
    }
}

// ---- SGD step in two launches (opt-in, ddrl_graphnet_train_step) ----------------------------------------------------------
// The three-kernel step (forward 125 us, loss, row-per-CTA backward 520 us per 16 384 rows) recomputes the forward inside
// the backward with two block barriers per row.  Split by what parallelises how:
//   K1 graphnet_train_fwd_kernel   one WARP per row (the forward kernel above) + the row's PPO loss gradient + the backward
//                                  down to the layer inputs; leaves per (net, row) a record {x_idx, mean of senders, dpre, y,
//                                  dpx[node], dout} in a workspace (2.1 KB; L2 / HBM streamed once) and per-CTA loss statistics;
//   K2 graphnet_train_acc_kernel   the weight gradients are rank-1 updates summed over rows: thread (h, fs) owns fixed
//                                  register accumulators (the layout of graphnet_kernel<true>) and streams the records with
//                                  no barrier in the row loop; it re-evaluates only ITS 5 hyper-network columns per node.
// Arithmetic per element is that of graphnet_kernel<true> + ppo_loss_grad_kernel.
constexpr int GTR_XI = 0, GTR_XM = GH, GTR_DPRE = 2 * GH, GTR_Y = 3 * GH, GTR_DPX = 4 * GH, GTR_DOUT = 8 * GH;
constexpr int GTR_REC = 8 * GH + GMAXO;       // 528 floats per (net, row)
constexpr int GWS = GH + 1;                   // padded stride of Wu / Wm: conflict-free by row AND by column
constexpr int GTF_SMEM_FLOATS = GE * GF * GH + GF * GH + 2 * GH * GWS + GH * GWF_WO + GMAXO +
                                GWF_WARPS * (GWF_ROW + GN * GH + 2 * GMAXO);

__global__ void __launch_bounds__(GWF_NT, 2)
graphnet_train_fwd_kernel(const float* __restrict__ theta, const int32_t* __restrict__ node_idx,
                          const float* __restrict__ state, const float* __restrict__ adj,
                          const float* __restrict__ actions, const float* __restrict__ old_logits,
                          const float* __restrict__ old_logp, const float* __restrict__ vf_preds,
                          const float* __restrict__ adv, const float* __restrict__ vtarg, int64_t B, int A,
                          const float* __restrict__ kl_coeff, const ddrl_ppo_hyper hp, float* __restrict__ rec,
                          double* __restrict__ stat_part) {
    extern __shared__ __align__(16) float gsm[];
    __shared__ double sStat[GWF_WARPS][DDRL_NSTAT];
    float* sWe = gsm;
    float* sbe = sWe + GE * GF * GH;
    float* sWu = sbe + GF * GH;                 // [GH][GWS]
    float* sWm = sWu + GH * GWS;
    float* sWo = sWm + GH * GWS;                // [GH][GWF_WO]
    float* sbo = sWo + GH * GWF_WO;
    float* sRowAll = sbo + GMAXO;               // [warps][GWF_ROW]
    float* sXAll = sRowAll + GWF_WARPS * GWF_ROW;   // [warps][GN][GH]
    float* sOAll = sXAll + GWF_WARPS * GN * GH;     // [warps][2][GMAXO]: model outputs, their loss gradient

    const int net = blockIdx.y;
    const int O = net == 0 ? 2 * A : 1;
    const GnOffsets o = gn_offsets(O);
    const float* th = theta + (net == 0 ? 0 : gn_offsets(2 * A).NP);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    for (int i = tid; i < GE * GF * GH; i += GWF_NT) sWe[i] = th[o.We + i];
    for (int i = tid; i < GF * GH; i += GWF_NT) sbe[i] = th[o.be + i];
    for (int i = tid; i < GH * GH; i += GWF_NT) {
        const int r = i >> 6, c = i & 63;
        sWu[r * GWS + c] = th[o.Wu + i];
        sWm[r * GWS + c] = th[o.Wm + i];
    }
    for (int i = tid; i < GH * GMAXO; i += GWF_NT) {
        const int hh = i / GMAXO, q = i - hh * GMAXO;
        sWo[hh * GWF_WO + q] = q < O ? th[o.Wo + hh * O + q] : 0.f;
    }
    if (tid < GMAXO) sbo[tid] = tid < O ? th[o.bo + tid] : 0.f;
    __syncthreads();

    float* sRow = sRowAll + warp * GWF_ROW;
    float* sX = sXAll + warp * GN * GH;
    float* sO = sOAll + warp * 2 * GMAXO;
    float* sDo = sO + GMAXO;
    float* recn = rec + (int64_t)net * B * GTR_REC;
    const float klc = kl_coeff[0];
    double acc[DDRL_NSTAT];
#pragma unroll
    for (int i = 0; i < DDRL_NSTAT; ++i) acc[i] = 0.0;

    const int64_t stride = (int64_t)gridDim.x * GWF_WARPS;
    for (int64_t b = (int64_t)blockIdx.x * GWF_WARPS + warp; b < B; b += stride) {
        for (int i = lane; i < GN * GS; i += 32) sRow[i] = state[b * GN * GS + i];
        if (lane < GN * GN) sRow[GN * GS + lane] = adj[b * GN * GN + lane];
        if (lane == GN * GN) sRow[GN * GS + GN * GN] = __int_as_float(node_idx[b]);
        __syncwarp();
        const GnRow g = gn_row(sRow);

        // ---- forward: identical to graphnet_fwd_warp_kernel -------------------------------------------------------------
        float e[GN][GE], a0[GN], a1[GN];
#pragma unroll
        for (int n = 0; n < GN; ++n) {
            a0[n] = 0.f;
            a1[n] = 0.f;
#pragma unroll
            for (int q = 0; q < GE; ++q) e[n][q] = sRow[n * GS + GF + q];
        }
#pragma unroll
        for (int f = 0; f < GF; ++f) {
            const int j = f * GH + lane;
            const float b0 = sbe[j], b1 = sbe[j + 32];
            const float w00 = sWe[j], w01 = sWe[j + 32];
            const float w10 = sWe[GF * GH + j], w11 = sWe[GF * GH + j + 32];
            const float w20 = sWe[2 * GF * GH + j], w21 = sWe[2 * GF * GH + j + 32];
            const float w30 = sWe[3 * GF * GH + j], w31 = sWe[3 * GF * GH + j + 32];
#pragma unroll
            for (int n = 0; n < GN; ++n) {
                if (g.need[n]) {
                    float p0 = b0, p1 = b1;
                    p0 = fmaf(e[n][0], w00, p0);
                    p1 = fmaf(e[n][0], w01, p1);
                    p0 = fmaf(e[n][1], w10, p0);
                    p1 = fmaf(e[n][1], w11, p1);
                    p0 = fmaf(e[n][2], w20, p0);
                    p1 = fmaf(e[n][2], w21, p1);
                    p0 = fmaf(e[n][3], w30, p0);
                    p1 = fmaf(e[n][3], w31, p1);
                    const float sf = sRow[n * GS + f];
                    a0[n] = fmaf(sf, gn_tanh(p0), a0[n]);
                    a1[n] = fmaf(sf, gn_tanh(p1), a1[n]);
                }
            }
        }
#pragma unroll
        for (int n = 0; n < GN; ++n) {
            if (g.need[n]) {
                sX[n * GH + lane] = gn_tanh(a0[n]);
                sX[n * GH + lane + 32] = gn_tanh(a1[n]);
            }
        }
        __syncwarp();
        const float inv_cnt = g.cnt > 0 ? 1.f / (float)g.cnt : 0.f;
        {
            float m0 = 0.f, m1 = 0.f;
#pragma unroll
            for (int n = 0; n < GN; ++n)
                if (g.is_snd[n]) {
                    m0 += sX[n * GH + lane];
                    m1 += sX[n * GH + lane + 32];
                }
            sRow[lane] = m0 * inv_cnt;              // xm in sRow[0..64); sRow[64..128) will take dpre
            sRow[lane + 32] = m1 * inv_cnt;
        }
        __syncwarp();
        const float* xs = sX + g.idx * GH;
        float y0 = 0.f, y1 = 0.f;
#pragma unroll 8
        for (int hh = 0; hh < GH; ++hh) {
            const float xi = xs[hh];
            const float xm = sRow[hh];
            y0 = fmaf(xi, sWu[hh * GWS + lane], y0);
            y1 = fmaf(xi, sWu[hh * GWS + lane + 32], y1);
            y0 = fmaf(xm, sWm[hh * GWS + lane], y0);
            y1 = fmaf(xm, sWm[hh * GWS + lane + 32], y1);
        }
        y0 = gn_tanh(y0);
        y1 = gn_tanh(y1);
#pragma unroll
        for (int q = 0; q < GMAXO; ++q) {
            if (q < O) {
                float v = fmaf(y0, sWo[lane * GWF_WO + q], y1 * sWo[(lane + 32) * GWF_WO + q]);
#pragma unroll
                for (int sft = 16; sft > 0; sft >>= 1) v += __shfl_xor_sync(0xffffffffu, v, sft);
                if (lane == q) sO[q] = v + sbo[q];
            }
        }
        __syncwarp();

        // ---- PPO loss gradient of this row w.r.t. this net's outputs (policy part: actor CTAs, value part: critic CTAs) --
        if (lane == 0) {
            double s[DDRL_NSTAT];
#pragma unroll
            for (int i = 0; i < DDRL_NSTAT; ++i) s[i] = 0.0;
            if (net == 0)
                ppo_row_policy(sO, A, actions + b * A, old_logits + b * 2 * A, old_logp[b], adv[b], klc, hp.clip_param,
                               hp.entropy_coeff, hp.inv_global_mb, sDo, s);
            else
                sDo[0] = ppo_row_value(sO[0], vf_preds[b], vtarg[b], hp.vf_clip_param, hp.vf_loss_coeff, hp.inv_global_mb, s);
#pragma unroll
            for (int i = 0; i < DDRL_NSTAT; ++i) acc[i] += s[i];
        }
        __syncwarp();

        // ---- backward to the layer inputs ---------------------------------------------------------------------------------
        float dy0 = 0.f, dy1 = 0.f;
#pragma unroll
        for (int q = 0; q < GMAXO; ++q) {
            if (q < O) {
                const float d = sDo[q];
                dy0 = fmaf(d, sWo[lane * GWF_WO + q], dy0);
                dy1 = fmaf(d, sWo[(lane + 32) * GWF_WO + q], dy1);
            }
        }
        const float dp0 = dy0 * (1.f - y0 * y0), dp1 = dy1 * (1.f - y1 * y1);
        float* rr = recn + b * GTR_REC;
        rr[GTR_XI + lane] = xs[lane];
        rr[GTR_XI + lane + 32] = xs[lane + 32];
        rr[GTR_XM + lane] = sRow[lane];
        rr[GTR_XM + lane + 32] = sRow[lane + 32];
        rr[GTR_DPRE + lane] = dp0;
        rr[GTR_DPRE + lane + 32] = dp1;
        rr[GTR_Y + lane] = y0;
        rr[GTR_Y + lane + 32] = y1;
        if (lane < GMAXO) rr[GTR_DOUT + lane] = lane < O ? sDo[lane] : 0.f;
        sRow[64 + lane] = dp0;
        sRow[96 + lane] = dp1;
        __syncwarp();
        float dxi0 = 0.f, dxi1 = 0.f, dxm0 = 0.f, dxm1 = 0.f;
#pragma unroll 8
        for (int hh = 0; hh < GH; ++hh) {
            const float d = sRow[64 + hh];
            dxi0 = fmaf(sWu[lane * GWS + hh], d, dxi0);
            dxi1 = fmaf(sWu[(lane + 32) * GWS + hh], d, dxi1);
            dxm0 = fmaf(sWm[lane * GWS + hh], d, dxm0);
            dxm1 = fmaf(sWm[(lane + 32) * GWS + hh], d, dxm1);
        }
        dxm0 *= inv_cnt;
        dxm1 *= inv_cnt;
#pragma unroll
        for (int n = 0; n < GN; ++n) {
            float q0 = 0.f, q1 = 0.f;
            if (g.need[n]) {
                const float dx0 = (n == g.idx ? dxi0 : 0.f) + (g.is_snd[n] ? dxm0 : 0.f);
                const float dx1 = (n == g.idx ? dxi1 : 0.f) + (g.is_snd[n] ? dxm1 : 0.f);
                const float x0 = sX[n * GH + lane], x1 = sX[n * GH + lane + 32];
                q0 = dx0 * (1.f - x0 * x0);
                q1 = dx1 * (1.f - x1 * x1);
            }
            rr[GTR_DPX + n * GH + lane] = q0;
            rr[GTR_DPX + n * GH + lane + 32] = q1;
        }
        __syncwarp();      // every lane is done with sRow / sX / sO before the next row overwrites them
    }

    if (lane == 0)
#pragma unroll
        for (int i = 0; i < DDRL_NSTAT; ++i) sStat[warp][i] = acc[i];
    __syncthreads();
    if (tid < DDRL_NSTAT) {
        double t = 0.0;
        for (int w = 0; w < GWF_WARPS; ++w) t += sStat[w][tid];
        stat_part[((int64_t)net * gridDim.x + blockIdx.x) * DDRL_NSTAT + tid] = t;
    }
}

__global__ void __launch_bounds__(GT2, 1)
graphnet_train_acc_kernel(const float* __restrict__ theta, const int32_t* __restrict__ node_idx,
                          const float* __restrict__ state, const float* __restrict__ adj, const float* __restrict__ rec,
                          int64_t B, int A, float* __restrict__ grad_part) {
    const int net = blockIdx.y;
    const int O = net == 0 ? 2 * A : 1;
    const GnOffsets oa = gn_offsets(2 * A);
    const GnOffsets o = gn_offsets(O);
    const int net_base = net == 0 ? 0 : oa.NP;
    const float* th = theta + net_base;
    const int tid = threadIdx.x, h = tid & (GH - 1), fs = tid >> 6;   // a warp = 32 consecutive hidden units, one fs
    const int G = gridDim.x, bx = blockIdx.x;

    float We[GK][GE], be[GK];
#pragma unroll
    for (int k = 0; k < GK; ++k) {
        const int f = fs + 4 * k;
        const bool ok = f < GF;
#pragma unroll
        for (int q = 0; q < GE; ++q) We[k][q] = ok ? th[o.We + q * GF * GH + f * GH + h] : 0.f;
        be[k] = ok ? th[o.be + f * GH + h] : 0.f;
    }
    float gWe[GK][GE], gbe[GK], gWu[16], gWm[16], gWo[GMAXO], gbo = 0.f;
#pragma unroll
    for (int k = 0; k < GK; ++k) {
        gbe[k] = 0.f;
#pragma unroll
        for (int q = 0; q < GE; ++q) gWe[k][q] = 0.f;
    }
#pragma unroll
    for (int i = 0; i < 16; ++i) { gWu[i] = 0.f; gWm[i] = 0.f; }
#pragma unroll
    for (int q = 0; q < GMAXO; ++q) gWo[q] = 0.f;

    const float* recn = rec + (int64_t)net * B * GTR_REC;
    for (int64_t b = bx; b < B; b += G) {
        const float* rr = recn + b * GTR_REC;
        const int idx = min(max(node_idx[b], 0), GN - 1);
        const float dpre = rr[GTR_DPRE + h], y = rr[GTR_Y + h];
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            gWu[i] = fmaf(rr[GTR_XI + 4 * i + fs], dpre, gWu[i]);
            gWm[i] = fmaf(rr[GTR_XM + 4 * i + fs], dpre, gWm[i]);
        }
#pragma unroll
        for (int q = 0; q < GMAXO; ++q)
            if (q < O) gWo[q] = fmaf(y, rr[GTR_DOUT + q], gWo[q]);
        if (tid < O) gbo += rr[GTR_DOUT + tid];
#pragma unroll
        for (int n = 0; n < GN; ++n) {
            const bool need = n == idx || adj[b * GN * GN + n * GN + idx] != 0.f;      // block-uniform
            if (need) {
                const float dpx = rr[GTR_DPX + n * GH + h];
                const float* st = state + b * GN * GS + n * GS;
                const float e0 = st[GF], e1 = st[GF + 1], e2 = st[GF + 2], e3 = st[GF + 3];
#pragma unroll
                for (int k = 0; k < GK; ++k) {
                    const int f = fs + 4 * k;
                    if (f < GF) {
                        float pre = be[k];
                        pre = fmaf(e0, We[k][0], pre);
                        pre = fmaf(e1, We[k][1], pre);
                        pre = fmaf(e2, We[k][2], pre);
                        pre = fmaf(e3, We[k][3], pre);
                        const float w = gn_tanh(pre);
                        const float dpw = dpx * st[f] * (1.f - w * w);
                        gWe[k][0] = fmaf(e0, dpw, gWe[k][0]);
                        gWe[k][1] = fmaf(e1, dpw, gWe[k][1]);
                        gWe[k][2] = fmaf(e2, dpw, gWe[k][2]);
                        gWe[k][3] = fmaf(e3, dpw, gWe[k][3]);
                        gbe[k] += dpw;
                    }
                }
            }
        }
    }

    float* gp = grad_part + (int64_t)bx * ((oa.NP + gn_offsets(1).NP + 3) & ~3) + net_base;
#pragma unroll
    for (int k = 0; k < GK; ++k) {
        const int f = fs + 4 * k;
        if (f < GF) {
#pragma unroll
            for (int q = 0; q < GE; ++q) gp[o.We + q * GF * GH + f * GH + h] = gWe[k][q];
            gp[o.be + f * GH + h] = gbe[k];
        }
    }
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        gp[o.Wu + (4 * i + fs) * GH + h] = gWu[i];
        gp[o.Wm + (4 * i + fs) * GH + h] = gWm[i];
    }
    if (fs == 0)
#pragma unroll
        for (int q = 0; q < GMAXO; ++q)
            if (q < O) gp[o.Wo + h * O + q] = gWo[q];
    if (tid < O) gp[o.bo + tid] = gbo;
}

// ---- GCN layer: y[b][n][u] = act(sum_f (sum_m An[n][m] x[b][m][f]) W[f][u] + bias[u]) ---------------------
__global__ void gcn_forward_kernel(const float* __restrict__ x, const float* __restrict__ adj, const float* __restrict__ W,
                                   const float* __restrict__ bias, int64_t B, int F, int U, int act,
                                   float* __restrict__ y) {
    extern __shared__ float sg[];   // ax[GN][F] per row handled by this CTA iteration
    __shared__ float sAn[GN][GN];
    for (int64_t b = blockIdx.x; b < B; b += gridDim.x) {
        __syncthreads();
        if (threadIdx.x < GN * GN) {
            const int n = threadIdx.x / GN;
            float d = 0.f;
            for (int m = 0; m < GN; ++m) d += adj[b * GN * GN + n * GN + m];
            // graph_ops.adj_norm: rowsum ** -1 (inf for isolated nodes, as in the reference)
            sAn[n][threadIdx.x % GN] = (1.f / d) * adj[b * GN * GN + threadIdx.x];
        }
        __syncthreads();
        for (int i = threadIdx.x; i < GN * F; i += blockDim.x) {
            const int n = i / F, f = i - n * F;
            float s = 0.f;
            for (int m = 0; m < GN; ++m) s = fmaf(sAn[n][m], x[(b * GN + m) * F + f], s);
            sg[i] = s;
        }
        __syncthreads();
        for (int i = threadIdx.x; i < GN * U; i += blockDim.x) {
            const int n = i / U, u = i - n * U;
            float s = 0.f;
            for (int f = 0; f < F; ++f) s = fmaf(sg[n * F + f], W[f * U + u], s);
            if (bias) s += bias[u];
            y[(b * GN + n) * U + u] = act == 1 ? tanhf(s) : s;
        }
    }
}

}  // namespace ddrl

using namespace ddrl;

extern "C" int ddrl_graphnet_num_params(int num_outputs) {
    if (num_outputs < 2 || num_outputs > GMAXO || (num_outputs & 1)) return DDRL_E_UNSUPPORTED_SHAPE;
    return gn_offsets(num_outputs).NP + gn_offsets(1).NP;
}

// forward schedule: 0 = one row per CTA (graphnet_kernel<false>), 1 = one row per warp (graphnet_fwd_warp_kernel);
// -1 = default, which the environment variable DDRL_GN_FWD_VARIANT may override (A/B timing without a rebuild)
static int g_gn_fwd_variant = -1;
constexpr int GN_FWD_DEFAULT = 1;   // measured: configs[3] iteration 75.5 -> 47.5 ms (profiles/README.md)
static int gn_fwd_variant() {
    if (g_gn_fwd_variant >= 0) return g_gn_fwd_variant;
    static int from_env = [] {
        const char* e = getenv("DDRL_GN_FWD_VARIANT");
        return (e && (e[0] == '0' || e[0] == '1') && e[1] == 0) ? e[0] - '0' : GN_FWD_DEFAULT;
    }();
    return from_env;
}

static int gn_ctas(int64_t B) {
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return (int)std::max<int64_t>(1, std::min<int64_t>(B, sms / 2));
}

// One launch of graphnet_fwd_warp_kernel<SAMPLE> (forward schedule 1).  B >= 1.
template <bool SAMPLE>
static int launch_fwd_warp(const float* theta, const int32_t* node_idx, const float* state, const float* adj,
                           const float* eps, int64_t B, int A, float* logits, float* value, float* action, float* logp,
                           void* stream, const char* who) {
    static bool attr_set = false;       // per process and instantiation; the attribute is sticky for the function
    const size_t smem = (size_t)GWF_SMEM_FLOATS * sizeof(float);
    if (!attr_set) {
        cudaError_t e = cudaFuncSetAttribute(graphnet_fwd_warp_kernel<SAMPLE>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             (int)smem);
        DDRL_REQUIRE(e == cudaSuccess, DDRL_E_CUDA, "%s: cudaFuncSetAttribute: %s", who, cudaGetErrorString(e));
        attr_set = true;
    }
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    // 3 CTAs per SM, the two nets side by side: (3 * sms / 2) CTAs per net, never more than one warp per row
    const int gx = (int)std::max<int64_t>(1, std::min<int64_t>((B + GWF_WARPS - 1) / GWF_WARPS, 3 * sms / 2));
    graphnet_fwd_warp_kernel<SAMPLE><<<dim3(gx, 2), GWF_NT, smem, (cudaStream_t)stream>>>(theta, node_idx, state, adj, B, A,
                                                                                         logits, value, eps, action, logp);
    DDRL_CHECK_LAUNCH(who);
    return DDRL_OK;
}

extern "C" int ddrl_graphnet_forward(const float* theta, const int32_t* node_idx, const float* state, const float* adj,
                                     int64_t B, int A, float* logits, float* value, void* stream) {
    DDRL_REQUIRE(theta && node_idx && state && adj && logits && value && B >= 0, DDRL_E_BADARG,
                 "graphnet_forward: null pointer or bad B");
    DDRL_REQUIRE(A >= 1 && A <= DDRL_MAX_ACT, DDRL_E_UNSUPPORTED_SHAPE, "graphnet_forward: unsupported A=%d", A);
    if (B == 0) return DDRL_OK;
    if (gn_fwd_variant() == 1)
        return launch_fwd_warp<false>(theta, node_idx, state, adj, nullptr, B, A, logits, value, nullptr, nullptr, stream,
                                      "graphnet_forward");
    graphnet_kernel<false><<<dim3(gn_ctas(B), 2), GT2, 0, (cudaStream_t)stream>>>(theta, node_idx, state, adj, nullptr,
                                                                                 nullptr, B, A, logits, value, nullptr);
    DDRL_CHECK_LAUNCH("graphnet_forward");
    return DDRL_OK;
}

extern "C" int ddrl_graphnet_act(const float* theta, const int32_t* node_idx, const float* state, const float* adj,
                                 const float* eps, int64_t B, int A, float* logits, float* value, float* action, float* logp,
                                 void* stream) {
    DDRL_REQUIRE(theta && node_idx && state && adj && eps && logits && value && action && logp && B >= 0, DDRL_E_BADARG,
                 "graphnet_act: null pointer or bad B");
    DDRL_REQUIRE(A >= 1 && A <= DDRL_MAX_ACT, DDRL_E_UNSUPPORTED_SHAPE, "graphnet_act: unsupported A=%d", A);
    if (B == 0) return DDRL_OK;
    return launch_fwd_warp<true>(theta, node_idx, state, adj, eps, B, A, logits, value, action, logp, stream, "graphnet_act");
}

// The variant selects the schedule of ddrl_graphnet_forward only; ddrl_graphnet_act always runs schedule 1.
extern "C" int ddrl_graphnet_set_variant(int variant) {
    DDRL_REQUIRE(variant >= -1 && variant <= 1, DDRL_E_BADARG, "graphnet_set_variant: variant must be -1 (default), 0 or 1");
    g_gn_fwd_variant = variant;
    return DDRL_OK;
}

extern "C" int ddrl_graphnet_backward(const float* theta, const int32_t* node_idx, const float* state, const float* adj,
                                      const float* dlogits, const float* dvalue, int64_t B, int A, int ctas,
                                      float* grad_part, void* stream) {
    DDRL_REQUIRE(theta && node_idx && state && adj && dlogits && dvalue && grad_part && B >= 1 && ctas >= 1,
                 DDRL_E_BADARG, "graphnet_backward: null pointer or bad B/ctas");
    DDRL_REQUIRE(A >= 1 && A <= DDRL_MAX_ACT, DDRL_E_UNSUPPORTED_SHAPE, "graphnet_backward: unsupported A=%d", A);
    graphnet_kernel<true><<<dim3(ctas, 2), GT2, 0, (cudaStream_t)stream>>>(theta, node_idx, state, adj, dlogits, dvalue, B,
                                                                          A, nullptr, nullptr, grad_part);
    DDRL_CHECK_LAUNCH("graphnet_backward");
    return DDRL_OK;
}

static int gn_train_fwd_ctas(int64_t B) {
    int dev = 0, sms = 148;
    if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return (int)std::max<int64_t>(1, std::min<int64_t>((B + GWF_WARPS - 1) / GWF_WARPS, sms));   // 2 CTAs per SM over the two nets
}

extern "C" int64_t ddrl_graphnet_train_ws_bytes(int64_t B) {
    return B < 0 ? DDRL_E_BADARG : 2 * B * (int64_t)GTR_REC * (int64_t)sizeof(float);
}

extern "C" int ddrl_graphnet_train_stat_parts(int64_t B) {
    return B < 1 ? DDRL_E_BADARG : 2 * gn_train_fwd_ctas(B);
}

extern "C" int ddrl_graphnet_train_step(const float* theta, const int32_t* node_idx, const float* state, const float* adj,
                                        const float* actions, const float* old_logits, const float* old_logp,
                                        const float* vf_preds, const float* adv, const float* vtarg, int64_t B, int A,
                                        const float* kl_coeff, const ddrl_ppo_hyper* hyper, int ctas, void* ws,
                                        float* grad_part, double* stat_part, void* stream) {
    DDRL_REQUIRE(theta && node_idx && state && adj && actions && old_logits && old_logp && vf_preds && adv && vtarg &&
                     kl_coeff && hyper && ws && grad_part && stat_part,
                 DDRL_E_BADARG, "graphnet_train_step: null pointer");
    DDRL_REQUIRE(B >= 1 && ctas >= 1, DDRL_E_BADARG, "graphnet_train_step: bad B/ctas");
    DDRL_REQUIRE(A >= 1 && A <= DDRL_MAX_ACT, DDRL_E_UNSUPPORTED_SHAPE, "graphnet_train_step: unsupported A=%d", A);
    static bool attr_set = false;
    const size_t smem = (size_t)GTF_SMEM_FLOATS * sizeof(float);
    if (!attr_set) {
        cudaError_t e = cudaFuncSetAttribute(graphnet_train_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        DDRL_REQUIRE(e == cudaSuccess, DDRL_E_CUDA, "graphnet_train_step: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
        attr_set = true;
    }
    cudaStream_t st = (cudaStream_t)stream;
    graphnet_train_fwd_kernel<<<dim3(gn_train_fwd_ctas(B), 2), GWF_NT, smem, st>>>(
        theta, node_idx, state, adj, actions, old_logits, old_logp, vf_preds, adv, vtarg, B, A, kl_coeff, *hyper,
        static_cast<float*>(ws), stat_part);
    DDRL_CHECK_LAUNCH("graphnet_train_step (forward + loss)");
    graphnet_train_acc_kernel<<<dim3(ctas, 2), GT2, 0, st>>>(theta, node_idx, state, adj, static_cast<const float*>(ws), B, A,
                                                            grad_part);
    DDRL_CHECK_LAUNCH("graphnet_train_step (weight gradients)");
    return DDRL_OK;
}

extern "C" int ddrl_gcn_forward(const float* x, const float* adj, const float* W, const float* b, int64_t B, int F,
                                int U, int act, float* y, void* stream) {
    DDRL_REQUIRE(x && adj && W && y && B >= 0 && F >= 1 && U >= 1, DDRL_E_BADARG, "gcn_forward: null pointer or bad shape");
    DDRL_REQUIRE(F <= 2048 && (act == 0 || act == 1), DDRL_E_UNSUPPORTED_SHAPE, "gcn_forward: F=%d > 2048 or act=%d", F, act);
    if (B == 0) return DDRL_OK;
    const int nb = (int)std::min<int64_t>(B, 148 * 8);
    gcn_forward_kernel<<<nb, 128, (size_t)GN * F * sizeof(float), (cudaStream_t)stream>>>(x, adj, W, b, B, F, U, act, y);
    DDRL_CHECK_LAUNCH("gcn_forward");
    return DDRL_OK;
}

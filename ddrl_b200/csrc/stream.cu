// HBM-bound streaming kernels of the learner path: MeanStdFilter update, GAE reverse scan,
// advantage standardisation, row shuffle, fixed-order gradient reduction, clip + TF1-Adam.
// All reductions use a fixed order (no float atomics) => bit-reproducible.
#include <algorithm>
#include <stdarg.h>
#include <string.h>

#include "common.cuh"
#include "fcnet_layout.cuh"
#include "fcnet_tc_layout.cuh"
#include <cuda_fp16.h>
#include "ppo_loss.cuh"
#include "sgd_tail.cuh"

namespace ddrl {

static thread_local char g_err[512] = "";
static int64_t g_launches = 0;
void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
void count_launch(int n) { __atomic_add_fetch(&g_launches, (int64_t)n, __ATOMIC_RELAXED); }

// =================================================================================================
// K4: MeanStdFilter — per-CTA (n, mean, M2) over a contiguous row range, then a fixed-order Chan merge
// =================================================================================================
constexpr int FT = 256;        // threads
constexpr int FROWS = 128;     // rows staged in shared memory per sub-chunk
constexpr int FMAXBLK = 256;   // partials per policy (64 until round 2: 16 dependent sub-chunks per CTA made the kernel latency bound,
                               // 75 us for 40 MB; the merge below is two-level so that its serial chain stays short)
constexpr int FMG = 16;        // merge groups: group g folds a contiguous run of partials, then the groups are folded in order
constexpr int FMAXCOL = DDRL_MAX_OBS / 8;  // columns per warp

struct Stat { double n, mean, m2; };
__device__ __forceinline__ void chan_merge(Stat& a, const Stat& b) {
    // RunningStat.update (ray.rllib.utils.filter): delta = M1 - M2; M = (n1 M1 + n2 M2)/n; S += S2 + delta^2 n1 n2 / n
    const double n = a.n + b.n;
    if (n == 0.0) return;
    const double delta = a.mean - b.mean;
    a.mean = (a.n * a.mean + b.n * b.mean) / n;
    a.m2 = a.m2 + b.m2 + delta * delta * a.n * b.n / n;
    a.n = n;
}

template <typename T>
__global__ void __launch_bounds__(FT) filter_partial_kernel(const T* __restrict__ x, int64_t R, int D, int nblk,
                                                            double* __restrict__ part) {
    extern __shared__ __align__(16) unsigned char fsm_raw[];
    T* xs = reinterpret_cast<T*>(fsm_raw);
    const int p = blockIdx.y, b = blockIdx.x, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t per = ((R + nblk - 1) / nblk + FROWS - 1) / FROWS * FROWS;
    const int64_t r0 = min((int64_t)b * per, R), r1 = min(r0 + per, R);
    const T* xp = x + (int64_t)p * R * D;
    Stat acc[FMAXCOL];
#pragma unroll
    for (int i = 0; i < FMAXCOL; ++i) acc[i] = Stat{0.0, 0.0, 0.0};
    for (int64_t c0 = r0; c0 < r1; c0 += FROWS) {
        const int nr = (int)min((int64_t)FROWS, r1 - c0);
        __syncthreads();
        for (int i = tid; i < nr * D; i += FT) xs[i] = xp[c0 * D + i];
        __syncthreads();
#pragma unroll
        for (int ci = 0; ci < FMAXCOL; ++ci) {
            const int d = warp + ci * 8;
            if (d < D) {
                double s = 0.0;
                for (int r = lane; r < nr; r += 32) s += (double)xs[r * D + d];
                s = warp_sum(s);
                const double mean = s / nr;
                double q = 0.0;
                for (int r = lane; r < nr; r += 32) {
                    const double e = (double)xs[r * D + d] - mean;
                    q = fma(e, e, q);
                }
                q = warp_sum(q);
                Stat c{(double)nr, mean, q};
                chan_merge(acc[ci], c);
            }
        }
    }
    if (lane == 0) {
#pragma unroll
        for (int ci = 0; ci < FMAXCOL; ++ci) {
            const int d = warp + ci * 8;
            if (d < D) {
                double* o = part + (((int64_t)p * nblk + b) * D + d) * 3;
                o[0] = acc[ci].n; o[1] = acc[ci].mean; o[2] = acc[ci].m2;
            }
        }
    }
}

__global__ void __launch_bounds__(FMG * 64) filter_merge_kernel(const double* __restrict__ part, int nblk, int D, int64_t R,
                                                                  int64_t* n_io, double* M, double* S, double* norm) {
    // thread (g, d): feature d, merge group g.  Fixed order: inside a group the partials in index order, then the groups in
    // order, then the running state — bit-reproducible; every thread's loads are independent of its merge chain's results, so
    // they are issued ahead (the one-level loop of round 1 waited for an L2 round trip per partial: 50 us for 64 partials).
    __shared__ Stat grp[FMG][64];
    const int p = blockIdx.x, d = threadIdx.x & 63, g = threadIdx.x >> 6;
    const int64_t n_old = n_io[p];
    const int64_t n_new = n_old + R;
    const int L = (nblk + FMG - 1) / FMG, i0 = g * L, i1 = min(nblk, i0 + L);
    Stat b{0.0, 0.0, 0.0};
    if (d < D) {
#pragma unroll 4
        for (int i = i0; i < i1; ++i) {
            const double* o = part + (((int64_t)p * nblk + i) * D + d) * 3;
            const Stat c{__ldg(o), __ldg(o + 1), __ldg(o + 2)};
            if (i == i0) b = c; else chan_merge(b, c);
        }
    }
    grp[g][d] = b;
    __syncthreads();  // also: every thread has read the old count before thread 0 overwrites it
    if (threadIdx.x == 0) n_io[p] = n_new;
    if (g != 0 || d >= D) return;
    for (int k = 1; k < FMG; ++k)
        if (grp[k][d].n != 0.0) chan_merge(b, grp[k][d]);      // (an empty group must not even round-trip (n mean) / n)
    Stat a{(double)n_old, M[p * D + d], S[p * D + d]};
    chan_merge(a, b);
    M[p * D + d] = a.mean;
    S[p * D + d] = a.m2;
    const double var = n_new > 1 ? a.m2 / (double)(n_new - 1) : a.mean * a.mean;
    norm[(int64_t)p * 2 * D + d] = a.mean;
    norm[(int64_t)p * 2 * D + D + d] = 1.0 / (sqrt(var) + 1e-8);
}

// =================================================================================================
// K5: GAE reverse scan (float64 like the reference's scipy.signal.lfilter on float64 deltas)
// =================================================================================================
constexpr int GT = 256;
__global__ void __launch_bounds__(GT) gae_kernel(const float* __restrict__ rewards, const float* __restrict__ values,
                                                 const uint8_t* __restrict__ dones, const float* __restrict__ v_boot,
                                                 int T, int64_t C, int cpe, double gamma, double lambda,
                                                 float* __restrict__ adv, float* __restrict__ vtarg,
                                                 double* __restrict__ part) {
    __shared__ double red[2][GT / 32];
    const int p = blockIdx.y;
    const int64_t c = (int64_t)blockIdx.x * GT + threadIdx.x;
    double s = 0.0, q = 0.0;
    if (c < C) {
        const int64_t base = (int64_t)p * T * C;
        const int64_t ce = c / cpe, Ce = C / cpe;
        double nv = (double)v_boot[(int64_t)p * C + c], na = 0.0;
        for (int t = T - 1; t >= 0; --t) {
            const double nd = dones[(int64_t)t * Ce + ce] ? 0.0 : 1.0;
            const double v = (double)values[base + (int64_t)t * C + c];
            const double delta = (double)rewards[base + (int64_t)t * C + c] + gamma * nd * nv - v;
            na = delta + gamma * lambda * nd * na;
            const float af = (float)na;
            adv[base + (int64_t)t * C + c] = af;
            vtarg[base + (int64_t)t * C + c] = (float)(na + v);
            s += (double)af;
            q = fma((double)af, (double)af, q);
            nv = v;
        }
    }
    s = warp_sum(s);
    q = warp_sum(q);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) { red[0][warp] = s; red[1][warp] = q; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double ss = 0.0, qq = 0.0;
        for (int i = 0; i < GT / 32; ++i) { ss += red[0][i]; qq += red[1][i]; }
        part[((int64_t)p * gridDim.x + blockIdx.x) * 2 + 0] = ss;
        part[((int64_t)p * gridDim.x + blockIdx.x) * 2 + 1] = qq;
    }
}

__global__ void gae_moments_kernel(const double* __restrict__ part, int nblk, double count, double* moments) {
    const int p = blockIdx.x;
    double s = 0.0, q = 0.0;
    // fixed assignment of partials to lanes, fixed tree afterwards
    for (int i = threadIdx.x; i < nblk; i += 32) { s += part[((int64_t)p * nblk + i) * 2]; q += part[((int64_t)p * nblk + i) * 2 + 1]; }
    s = warp_sum(s);
    q = warp_sum(q);
    if (threadIdx.x == 0) { moments[p * 3 + 0] = count; moments[p * 3 + 1] = s; moments[p * 3 + 2] = q; }
}

__global__ void adv_standardize_kernel(float* __restrict__ adv, const double* __restrict__ moments, int64_t R) {
    const int p = blockIdx.y;
    const double n = moments[p * 3], mean = moments[p * 3 + 1] / n;
    const double var = fmax(moments[p * 3 + 2] / n - mean * mean, 0.0);
    const float mf = (float)mean, sf = fmaxf(1e-4f, (float)sqrt(var));
    float* a = adv + (int64_t)p * R;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < R; i += (int64_t)gridDim.x * blockDim.x)
        a[i] = (a[i] - mf) / sf;
}

__global__ void gather_rows_kernel(const float* __restrict__ src, const int32_t* __restrict__ perm, int64_t R, int W,
                                   float* __restrict__ dst) {
    const int p = blockIdx.y;
    const float* s = src + (int64_t)p * R * W;
    float* d = dst + (int64_t)p * R * W;
    const int32_t* pm = perm + (int64_t)p * R;
    const int64_t n = R * W;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / W;
        const int c = (int)(i - r * W);
        d[i] = s[(int64_t)pm[r] * W + c];
    }
}

// =================================================================================================
// gradient partial reduce (fixed order) and K7: clip_by_global_norm + TF1 Adam
// =================================================================================================
__global__ void grad_reduce_kernel(const float* __restrict__ gpart, const double* __restrict__ spart, int G, int NP,
                                   float* __restrict__ grad, double* __restrict__ step_stats,
                                   const int32_t* __restrict__ step_ctr) {
    const int p = blockIdx.y, P = gridDim.y;
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    const int NPs = (NP + 3) & ~3;   // partial stride (ddrl_b200.h)
    if (j < NP) {
        const float* g = gpart + (int64_t)p * G * NPs + j;
        float s = 0.f;
#pragma unroll 4
        for (int i = 0; i < G; ++i) s += g[(int64_t)i * NPs];
        grad[(int64_t)p * NP + j] = s;
    }
    if (blockIdx.x == 0 && threadIdx.x < DDRL_NSTAT && spart && step_stats) {
        const int step = step_ctr ? *step_ctr : 0;
        double s = 0.0;
        for (int i = 0; i < G; ++i) s += spart[((int64_t)p * G + i) * DDRL_NSTAT + threadIdx.x];
        step_stats[((int64_t)step * P + p) * DDRL_NSTAT + threadIdx.x] = s;
    }
}

constexpr int AT = 256;
__global__ void __launch_bounds__(AT) clip_adam_kernel(float* __restrict__ theta, float* __restrict__ m,
                                                       float* __restrict__ v, float* beta_pow,
                                                       const float* __restrict__ grad, int NP, float lr, float beta1,
                                                       float beta2, float eps, float clip, float* gnorm_out,
                                                       int32_t* step_ctr, int32_t* sync_ws, float* __restrict__ img,
                                                       unsigned char* __restrict__ tcimg, int imgD, int imgA) {
    __shared__ float red[AT / 32];
    __shared__ float s_scale;
    const int p = blockIdx.y, P = gridDim.y, tid = threadIdx.x;
    const float* g = grad + (int64_t)p * NP;
    // every CTA of the policy recomputes the global norm in the same fixed order (identical bits everywhere)
    float ss = 0.f;
    for (int i = tid; i < NP; i += AT) ss = fmaf(g[i], g[i], ss);
    ss = warp_sum(ss);
    if ((tid & 31) == 0) red[tid >> 5] = ss;
    __syncthreads();
    if (tid == 0) {
        float t = 0.f;
        for (int i = 0; i < AT / 32; ++i) t += red[i];
        const float norm = sqrtf(t);
        // tf.clip_by_global_norm: scale = clip * min(1/norm, 1/clip)
        s_scale = clip > 0.f ? clip * fminf(1.f / norm, 1.f / clip) : 1.f;
        if (gnorm_out && blockIdx.x == 0) gnorm_out[p] = norm;
    }
    __syncthreads();
    const float scale = s_scale;
    const float b1p = beta_pow[p * 2], b2p = beta_pow[p * 2 + 1];
    // tensorflow/core/kernels/training_ops.cc ApplyAdam (non-nesterov)
    const float alpha = lr * sqrtf(1.f - b2p) / (1.f - b1p);
    const int j = blockIdx.x * AT + tid;
    if (j < NP) {
        const int64_t k = (int64_t)p * NP + j;
        const float gj = g[j] * scale;
        float mj = m[k], vj = v[k];
        mj += (gj - mj) * (1.f - beta1);
        vj += (gj * gj - vj) * (1.f - beta2);
        m[k] = mj;
        v[k] = vj;
        const float tnew = theta[k] - (mj * alpha) / (sqrtf(vj) + eps);
        theta[k] = tnew;
        if (img) {   // keep the packed shared-memory image of the FCNet weights in step with theta
            const FcSmem L = fc_smem(imgD, imgA, false);
            const FcOffsets o = fc_offsets(imgD, imgA);
            int p0, p1;
            fc_img_pos(L, o, imgD, imgA, j, p0, p1);
            float* im = img + (int64_t)p * L.x;
            im[p0] = tnew;
            if (p1 >= 0) im[p1] = tnew;
        }
        if (tcimg) {   // tensor-core image: fp16 (hi, lo) of 256*w for the GEMM weights, fp32 for biases / heads
            const TcImg L = tc_img(imgD, imgA);
            const FcOffsets o = fc_offsets(imgD, imgA);
            bool f16;
            int p0, p1;
            tc_img_pos(L, o, imgD, imgA, j, f16, p0, p1);
            unsigned char* im = tcimg + (int64_t)p * L.bytes;
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
    // arrival ticket: the last CTA advances the beta powers / step counter after everyone has read them
    __syncthreads();
    if (tid == 0) {
        __threadfence();
        const int total = gridDim.x * gridDim.y;
        const int t = atomicAdd(sync_ws, 1);
        if (t == total - 1) {
            for (int q = 0; q < P; ++q) {
                beta_pow[q * 2] *= beta1;
                beta_pow[q * 2 + 1] *= beta2;
            }
            if (step_ctr) *step_ctr += 1;
            *sync_ws = 0;
            __threadfence();
        }
    }
}

// K6 (stand-alone): PPO loss gradient w.r.t. model outputs, for models whose forward/backward are separate
// kernels (GraphNet).  grid (G, P); per-CTA stat partials like the fused FCNet kernel.
constexpr int LT = 256;
__global__ void __launch_bounds__(LT) ppo_loss_grad_kernel(
    const float* __restrict__ logits, const float* __restrict__ value, const float* __restrict__ actions,
    const float* __restrict__ old_logits, const float* __restrict__ old_logp, const float* __restrict__ vf_preds,
    const float* __restrict__ adv, const float* __restrict__ vtarg, int64_t R, int A, const float* __restrict__ kl_coeff,
    const ddrl_ppo_hyper hp, float* __restrict__ dlogits, float* __restrict__ dvalue, double* __restrict__ stat_part) {
    __shared__ double red[LT / 32][DDRL_NSTAT];
    const int p = blockIdx.y, A2 = 2 * A;
    const float klc = kl_coeff[p];
    double st[DDRL_NSTAT];
#pragma unroll
    for (int i = 0; i < DDRL_NSTAT; ++i) st[i] = 0.0;
    for (int64_t r = (int64_t)blockIdx.x * LT + threadIdx.x; r < R; r += (int64_t)gridDim.x * LT) {
        const int64_t gr = (int64_t)p * R + r;
        float out[2 * DDRL_MAX_ACT + 1], dl[2 * DDRL_MAX_ACT + 1];
        double s[DDRL_NSTAT];
#pragma unroll
        for (int i = 0; i < 2 * DDRL_MAX_ACT; ++i)
            if (i < A2) out[i] = logits[gr * A2 + i];
        out[A2] = value[gr];
        ppo_row_loss(out, A, actions + gr * A, old_logits + gr * A2, old_logp[gr], vf_preds[gr], adv[gr], vtarg[gr],
                     klc, hp, dl, s);
#pragma unroll
        for (int i = 0; i < 2 * DDRL_MAX_ACT; ++i)
            if (i < A2) dlogits[gr * A2 + i] = dl[i];
        dvalue[gr] = dl[A2];
#pragma unroll
        for (int i = 0; i < DDRL_NSTAT; ++i) st[i] += s[i];
    }
#pragma unroll
    for (int i = 0; i < DDRL_NSTAT; ++i) st[i] = warp_sum(st[i]);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0)
#pragma unroll
        for (int i = 0; i < DDRL_NSTAT; ++i) red[warp][i] = st[i];
    __syncthreads();
    if (threadIdx.x < DDRL_NSTAT) {
        double t = 0.0;
        for (int w = 0; w < LT / 32; ++w) t += red[w][threadIdx.x];
        stat_part[((int64_t)p * gridDim.x + blockIdx.x) * DDRL_NSTAT + threadIdx.x] = t;
    }
}

// a3: per-agent observation gather (quantruped_v3.get_obs_indices + distribute_observations): pure indexing
template <typename T>
__global__ void obs_gather_kernel(const T* __restrict__ full, int64_t S, int Dfull, const int32_t* __restrict__ table, int Ag,
                                  int D, int P, float* __restrict__ out) {
    const int k = Ag / P;
    const int64_t n = S * Ag * D;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int d = (int)(i % D);
        const int64_t t = i / D;
        const int a = (int)(t % Ag);
        const int64_t s = t / Ag;
        const int p = a / k, j = a - p * k;
        out[(((int64_t)p * S + s) * k + j) * D + d] = (float)full[s * Dfull + table[a * D + d]];
    }
}

// N2: node features of the shared-graph env, batched over env-steps (all arithmetic in float64 with explicit _rn
// operations so that no FMA contraction changes a bit against numpy):
//   state[s][a][d <  Dn] = clip((full[s][table[a][d]] - mean[..]) / (std[..] + 1e-8), -clip, clip)   (env filter, frozen stats)
//   state[s][a][Dn + 0..3] = full[s][1:5] (x) [0, 0, zw[a][0], zw[a][1]]                                  (leg_encoding_ego)
// With rep != 0 every env-step emits Ag sample rows (row = s*Ag + j carries the whole [Ag][Dn+4] matrix and node_idx = j),
// which is the batch layout RLlib builds from the per-agent observation tuples.
template <typename T>
__global__ void graph_obs_build_kernel(const T* __restrict__ full, int64_t S, int Dfull, const int32_t* __restrict__ table,
                                       int Ag, int Dn, const double* __restrict__ mean, const double* __restrict__ stdv,
                                       double clip, const double* __restrict__ zw, int rep, float* __restrict__ state,
                                       int32_t* __restrict__ node_idx) {
    const int F = Dn + 4;
    const int64_t n = S * Ag * F;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int d = (int)(i % F);
        const int64_t t = i / F;
        const int a = (int)(t % Ag);
        const int64_t s = t / Ag;
        const T* o = full + s * Dfull;
        double y;
        if (d < Dn) {
            const int c = table[a * Dn + d];
            y = (double)o[c];
            if (mean) y = __dsub_rn(y, mean[c]);
            if (stdv) y = __ddiv_rn(y, __dadd_rn(stdv[c], 1e-8));
            if (clip > 0.0) y = fmin(fmax(y, -clip), clip);
        } else {
            const double x1 = (double)o[1], y1 = (double)o[2], z1 = (double)o[3], w1 = (double)o[4];
            const double qz = zw[2 * a], qw = zw[2 * a + 1];
            // quat2 = (0, 0, qz, qw); the zero products are kept out: x + (+-0) == x for every x numpy can produce here
            switch (d - Dn) {
                case 0: y = __dadd_rn(__dmul_rn(x1, qw), __dmul_rn(y1, qz)); break;                      //  x1*w2 + y1*z2
                case 1: y = __dadd_rn(__dmul_rn(-x1, qz), __dmul_rn(y1, qw)); break;                     // -x1*z2 + y1*w2
                case 2: y = __dadd_rn(__dmul_rn(z1, qw), __dmul_rn(w1, qz)); break;                      //  z1*w2 + w1*z2
                default: y = __dadd_rn(__dmul_rn(-z1, qz), __dmul_rn(w1, qw)); break;                    // -z1*z2 + w1*w2
            }
        }
        const float v = (float)y;
        if (rep) {
            for (int j = 0; j < Ag; ++j) state[((s * Ag + j) * Ag + a) * F + d] = v;
            if (d == 0 && node_idx) node_idx[s * Ag + a] = a;
        } else {
            state[i] = v;
        }
    }
}

// N2: per-agent reward / cost split of the multi-agent adaptor, batched over env-steps (float64 arithmetic like numpy):
//   contact_a = sum_body Wc[a][body] * contact_w * sum_j clip(cfrc[body][j], -1, 1)^2      (distribute_contact_cost)
//   mode 0  fw / Ag - ctrl_w * |act_a|^2 - contact_a                                        (distribute_per_leg_reward)
//   mode 1  fw - Ag * (ctrl_w * |act_a|^2 + contact_a)                                      (… with norm_reward)
//   mode 2  (fw - ctrl_w * sum_a |act_a|^2 - contact_w * sum_all clip(cfrc)^2) / Ag         (distribute_global_reward)
//   mode 3  fw / Ag - ctrl_w * 0.25 * sum_a |act_a|^2 - contact_a                           (GlobalCosts env)
__global__ void reward_split_kernel(const float* __restrict__ fw, const float* __restrict__ act, const double* __restrict__ cfrc,
                                    const double* __restrict__ Wc, int64_t S, int Ag, int A, int NB, double ctrl_w,
                                    double contact_w, int mode, float* __restrict__ rew) {
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= S) return;
    double body[16];
    double all_contact = 0.0;
    for (int b = 0; b < NB; ++b) {
        double q = 0.0;
        for (int j = 0; j < 6; ++j) {
            const double f = fmin(fmax(cfrc[(s * NB + b) * 6 + j], -1.0), 1.0);
            q += contact_w * (f * f);
        }
        body[b] = q;
        all_contact += q;
    }
    double ctrl[8], ctrl_sum = 0.0;
    for (int a = 0; a < Ag; ++a) {
        double q = 0.0;
        for (int j = 0; j < A; ++j) {
            const double v = (double)act[(s * Ag + a) * A + j];
            q += v * v;
        }
        ctrl[a] = q;
        ctrl_sum += q;
    }
    const double f = (double)fw[s];
    for (int a = 0; a < Ag; ++a) {
        double c = 0.0;
        for (int b = 0; b < NB; ++b) c += body[b] * Wc[a * NB + b];
        double r;
        if (mode == 0) r = f / Ag - ctrl_w * ctrl[a] - c;
        else if (mode == 1) r = f - Ag * (ctrl_w * ctrl[a] + c);
        else if (mode == 2) r = (f - ctrl_w * ctrl_sum - all_contact) / Ag;
        else r = f / Ag - ctrl_w * 0.25 * ctrl_sum - c;
        rew[s * Ag + a] = (float)r;
    }
}

// N2: concatenate_actions (adaptor :205-212) with RLlib's clip_actions: env_action[table[a][j]] = clip(act[a][j], lo, hi)
__global__ void concat_actions_kernel(const float* __restrict__ act, const int32_t* __restrict__ table, int64_t S, int Ag, int A,
                                      int Afull, float lo, float hi, float* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= S * Ag * A) return;
    const int64_t s = i / (Ag * A);
    const int k = (int)(i % (Ag * A));
    out[s * Afull + table[k]] = fminf(fmaxf(act[i], lo), hi);
}

// DiagGaussian sample + logp (RLlib models/tf/tf_action_dist.py) for models without a fused epilogue.
__global__ void dg_sample_kernel(const float* __restrict__ logits, const float* __restrict__ eps, int64_t R, int A,
                                 float* __restrict__ action, float* __restrict__ logp) {
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < R; r += (int64_t)gridDim.x * blockDim.x)
        logp[r] = dg_sample_row(logits, eps, r, A, action);
}

__global__ void leg_coupling_kernel(float* __restrict__ logits, const int32_t* __restrict__ node_id,
                                    const float* __restrict__ coupling, int64_t B, int W) {
    const int64_t n = B * W;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t b = i / W;
        const int j = (int)(i - b * W);
        if (j < 2) logits[i] *= coupling[node_id[b] * 2 + j];
    }
}

// Optional FCNet layouts (vf_share_layers / free_log_std, models/fcnet_glorot_uniform_init.py:30-36,85-113) on the two-branch
// kernels: the kernels' parameter vector is an index-select of the model's variables (tied value-branch copies, constant
// zeros), and the model gradient is the fixed-order sum of the (at most two) kernel-layout gradients of each variable.
__global__ void param_expand_kernel(const float* __restrict__ theta_model, const int32_t* __restrict__ map, int NPm, int NPk,
                                    float* __restrict__ theta_kernel) {
    const int p = blockIdx.y;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < NPk; i += gridDim.x * blockDim.x) {
        const int j = map[i];
        theta_kernel[(int64_t)p * NPk + i] = (j >= 0 && j < NPm) ? theta_model[(int64_t)p * NPm + j] : 0.f;
    }
}
__global__ void grad_tie_kernel(const float* __restrict__ grad_kernel, const int32_t* __restrict__ inv, int NPm, int NPk,
                                float* __restrict__ grad_model) {
    const int p = blockIdx.y;
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < NPm; j += gridDim.x * blockDim.x) {
        const int i0 = inv[2 * j], i1 = inv[2 * j + 1];
        float g = i0 >= 0 ? grad_kernel[(int64_t)p * NPk + i0] : 0.f;
        if (i1 >= 0) g += grad_kernel[(int64_t)p * NPk + i1];
        grad_model[(int64_t)p * NPm + j] = g;
    }
}

// LegCoupling backward: dlogits_pre = dout * coeff (in place on dout) and dcoupling[n][j] = sum over rows b with
// node_id[b] == n of dout[b][j] * logits_pre[b][j], j < 2 (the trainable tf.Variable of the reference layer).
// ONE block, fixed-order tree reduction over float64 per-thread sums: bit-reproducible (the op is tiny next to the MLP).
__global__ void __launch_bounds__(1024, 1) leg_coupling_bwd_kernel(float* __restrict__ dout, const float* __restrict__ logits_pre,
                                                                   const int32_t* __restrict__ node_id,
                                                                   const float* __restrict__ coupling, int64_t B, int W,
                                                                   float* __restrict__ dcoupling) {
    __shared__ double red[32][8];
    double acc[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) acc[i] = 0.0;
    for (int64_t b = threadIdx.x; b < B; b += blockDim.x) {
        const int n = node_id[b] & 3;
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const float g = dout[b * W + j];
            const double prod = (double)g * (double)logits_pre[b * W + j];
#pragma unroll
            for (int q = 0; q < 4; ++q) acc[2 * q + j] += (q == n) ? prod : 0.0;
            dout[b * W + j] = g * coupling[n * 2 + j];
        }
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const double v = warp_sum(acc[i]);
        if (lane == 0) red[warp][i] = v;
    }
    __syncthreads();
    if (threadIdx.x < 8) {
        double v = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) v += red[w][threadIdx.x];
        dcoupling[threadIdx.x] = (float)v;
    }
}

}  // namespace ddrl

using namespace ddrl;

extern "C" const char* ddrl_last_error(void) { return g_err; }
extern "C" int ddrl_abi_version(void) { return 1; }
extern "C" int64_t ddrl_launch_count(void) { return __atomic_load_n(&g_launches, __ATOMIC_RELAXED); }

static int filter_nblk(int64_t R) {
    return (int)std::max<int64_t>(1, std::min<int64_t>(FMAXBLK, (R + FROWS - 1) / FROWS));
}

extern "C" int64_t ddrl_filter_ws_bytes(int P, int64_t R, int D) {
    return (int64_t)P * filter_nblk(R) * D * 3 * (int64_t)sizeof(double);
}

extern "C" int ddrl_filter_num_partials(int64_t R) { return filter_nblk(R); }

extern "C" int ddrl_filter_partial(const void* x, int x_is_f64, int P, int64_t R, int D, void* ws, void* stream) {
    DDRL_REQUIRE(ws && P >= 1 && R >= 0, DDRL_E_BADARG, "filter_partial: null workspace or bad P/R");
    DDRL_REQUIRE(R == 0 || x, DDRL_E_BADARG, "filter_partial: x is null");
    DDRL_REQUIRE(D >= 1 && D <= DDRL_MAX_OBS, DDRL_E_UNSUPPORTED_SHAPE, "filter_partial: D=%d > %d", D, DDRL_MAX_OBS);
    cudaStream_t st = (cudaStream_t)stream;
    const int nblk = filter_nblk(R);
    if (R == 0) {
        cudaMemsetAsync(ws, 0, (size_t)ddrl_filter_ws_bytes(P, R, D), st);
        return DDRL_OK;
    }
    dim3 grid(nblk, P);
    if (x_is_f64) {
        static bool attr = false;
        if (!attr) {
            cudaFuncSetAttribute(filter_partial_kernel<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
            attr = true;
        }
        filter_partial_kernel<double><<<grid, FT, (size_t)FROWS * D * sizeof(double), st>>>((const double*)x, R, D, nblk,
                                                                                           (double*)ws);
    } else {
        filter_partial_kernel<float><<<grid, FT, (size_t)FROWS * D * sizeof(float), st>>>((const float*)x, R, D, nblk,
                                                                                         (double*)ws);
    }
    DDRL_CHECK_LAUNCH("filter_partial");
    return DDRL_OK;
}

extern "C" int ddrl_filter_merge(const void* parts, int nparts, int P, int D, int64_t R_total, int64_t* n, double* M,
                                 double* S, double* norm, void* stream) {
    DDRL_REQUIRE(parts && n && M && S && norm && P >= 1 && nparts >= 0 && R_total >= 0, DDRL_E_BADARG,
                 "filter_merge: null pointer or bad shape");
    DDRL_REQUIRE(D >= 1 && D <= DDRL_MAX_OBS, DDRL_E_UNSUPPORTED_SHAPE, "filter_merge: D=%d > %d", D, DDRL_MAX_OBS);
    filter_merge_kernel<<<P, FMG * 64, 0, (cudaStream_t)stream>>>((const double*)parts, nparts, D, R_total, n, M, S, norm);
    DDRL_CHECK_LAUNCH("filter_merge");
    return DDRL_OK;
}

extern "C" int ddrl_filter_update(const void* x, int x_is_f64, int P, int64_t R, int D, int64_t* n, double* M,
                                  double* S, double* norm, void* ws, void* stream) {
    DDRL_REQUIRE(n && M && S && norm && ws, DDRL_E_BADARG, "filter_update: null pointer");
    const int rc = ddrl_filter_partial(x, x_is_f64, P, R, D, ws, stream);
    if (rc != DDRL_OK) return rc;
    return ddrl_filter_merge(ws, filter_nblk(R), P, D, R, n, M, S, norm, stream);
}

extern "C" int64_t ddrl_gae_ws_bytes(int P, int64_t C) { return (int64_t)P * ((C + GT - 1) / GT) * 2 * (int64_t)sizeof(double); }

extern "C" int ddrl_gae(const float* rewards, const float* values, const uint8_t* dones, const float* v_boot, int P,
                        int T, int64_t C, int cols_per_env, double gamma, double lambda, float* adv, float* vtarg,
                        double* moments, void* ws, void* stream) {
    DDRL_REQUIRE(rewards && values && dones && v_boot && adv && vtarg && moments && ws, DDRL_E_BADARG, "gae: null pointer");
    DDRL_REQUIRE(P >= 1 && T >= 1 && C >= 1 && cols_per_env >= 1 && C % cols_per_env == 0, DDRL_E_BADARG,
                 "gae: bad P/T/C/cols_per_env (C must be a multiple of cols_per_env)");
    cudaStream_t st = (cudaStream_t)stream;
    const int nblk = (int)((C + GT - 1) / GT);
    gae_kernel<<<dim3(nblk, P), GT, 0, st>>>(rewards, values, dones, v_boot, T, C, cols_per_env, gamma,
                                             lambda, adv, vtarg, (double*)ws);
    DDRL_CHECK_LAUNCH("gae");
    gae_moments_kernel<<<P, 32, 0, st>>>((const double*)ws, nblk, (double)T * (double)C, moments);
    DDRL_CHECK_LAUNCH("gae_moments");
    return DDRL_OK;
}

extern "C" int ddrl_adv_standardize(float* adv, const double* moments, int P, int64_t R, void* stream) {
    DDRL_REQUIRE(adv && moments && P >= 1 && R >= 1, DDRL_E_BADARG, "adv_standardize: null pointer or bad P/R");
    const int nb = (int)std::min<int64_t>(1024, (R + 255) / 256);
    adv_standardize_kernel<<<dim3(nb, P), 256, 0, (cudaStream_t)stream>>>(adv, moments, R);
    DDRL_CHECK_LAUNCH("adv_standardize");
    return DDRL_OK;
}

extern "C" int ddrl_gather_rows(const float* src, const int32_t* perm, int P, int64_t R, int W, float* dst, void* stream) {
    DDRL_REQUIRE(src && perm && dst && P >= 1 && R >= 1 && W >= 1, DDRL_E_BADARG, "gather_rows: null pointer or bad shape");
    DDRL_REQUIRE(src != dst, DDRL_E_BADARG, "gather_rows: in-place gather is not supported");
    const int nb = (int)std::min<int64_t>(2048, (R * W + 255) / 256);
    gather_rows_kernel<<<dim3(nb, P), 256, 0, (cudaStream_t)stream>>>(src, perm, R, W, dst);
    DDRL_CHECK_LAUNCH("gather_rows");
    return DDRL_OK;
}

extern "C" int ddrl_grad_reduce(const float* grad_part, const double* stat_part, int P, int G, int NP, float* grad,
                                double* step_stats, const int32_t* step_ctr, void* stream) {
    DDRL_REQUIRE(grad_part && grad && P >= 1 && G >= 1 && NP >= 1, DDRL_E_BADARG, "grad_reduce: null pointer or bad shape");
    grad_reduce_kernel<<<dim3((NP + 255) / 256, P), 256, 0, (cudaStream_t)stream>>>(grad_part, stat_part, G, NP, grad,
                                                                                   step_stats, step_ctr);
    DDRL_CHECK_LAUNCH("grad_reduce");
    return DDRL_OK;
}

extern "C" int ddrl_fcnet_train_supported(int D, int A, int tensor_cores) {
    if (tensor_cores)      // ddrl_ppo_train_step_tc: shape check, then its shared memory (branch-sequential kernel)
        return ddrl_fcnet_tc_image_bytes(D, A) > 0 && tc_smem(D, A).total <= 227 * 1024;
    // ddrl_ppo_train_step: shape check, then the train kernel's shared memory
    return D >= 1 && D <= DDRL_MAX_OBS && A >= 1 && A <= DDRL_MAX_ACT &&
           (size_t)fc_smem(D, A, false, true).total * sizeof(float) <= 227 * 1024;
}

extern "C" int ddrl_clip_adam(float* theta, float* m, float* v, float* beta_pow, const float* grad, int P, int NP,
                              float lr, float beta1, float beta2, float eps, float grad_clip, float* gnorm_out,
                              int32_t* step_ctr, int32_t* sync_ws, float* fcnet_img, void* fcnet_tc_img, int img_D,
                              int img_A, void* stream) {
    DDRL_REQUIRE(theta && m && v && beta_pow && grad && sync_ws && P >= 1 && NP >= 1, DDRL_E_BADARG,
                 "clip_adam: null pointer or bad shape");
    DDRL_REQUIRE(!(fcnet_img || fcnet_tc_img) || (img_D >= 1 && img_D <= DDRL_MAX_OBS && img_A >= 1 && img_A <= DDRL_MAX_ACT &&
                                fc_offsets(img_D, img_A).NP == NP),
                 DDRL_E_BADARG, "clip_adam: fcnet image given but (D=%d, A=%d) does not match NP=%d", img_D, img_A, NP);
    DDRL_REQUIRE(!fcnet_tc_img || ddrl_fcnet_tc_image_bytes(img_D, img_A) > 0, DDRL_E_UNSUPPORTED_SHAPE,
                 "clip_adam: no tensor-core image exists for D=%d A=%d (A in {1,2,4,8}, D <= 63)", img_D, img_A);
    clip_adam_kernel<<<dim3((NP + AT - 1) / AT, P), AT, 0, (cudaStream_t)stream>>>(
        theta, m, v, beta_pow, grad, NP, lr, beta1, beta2, eps, grad_clip, gnorm_out, step_ctr, sync_ws, fcnet_img,
        (unsigned char*)fcnet_tc_img, img_D, img_A);
    DDRL_CHECK_LAUNCH("clip_adam");
    return DDRL_OK;
}

extern "C" int ddrl_ppo_loss_grad(const float* logits, const float* value, const float* actions, const float* old_logits,
                                  const float* old_logp, const float* vf_preds, const float* adv, const float* vtarg,
                                  int P, int64_t R, int A, const float* kl_coeff, const ddrl_ppo_hyper* hyper, int ctas,
                                  float* dlogits, float* dvalue, double* stat_part, void* stream) {
    DDRL_REQUIRE(logits && value && actions && old_logits && old_logp && vf_preds && adv && vtarg && kl_coeff && hyper &&
                     dlogits && dvalue && stat_part,
                 DDRL_E_BADARG, "ppo_loss_grad: null pointer");
    DDRL_REQUIRE(P >= 1 && R >= 1 && ctas >= 1, DDRL_E_BADARG, "ppo_loss_grad: bad P/R/ctas");
    DDRL_REQUIRE(A >= 1 && A <= DDRL_MAX_ACT, DDRL_E_UNSUPPORTED_SHAPE, "ppo_loss_grad: unsupported A=%d", A);
    ppo_loss_grad_kernel<<<dim3(ctas, P), LT, 0, (cudaStream_t)stream>>>(logits, value, actions, old_logits, old_logp,
                                                                        vf_preds, adv, vtarg, R, A, kl_coeff, *hyper,
                                                                        dlogits, dvalue, stat_part);
    DDRL_CHECK_LAUNCH("ppo_loss_grad");
    return DDRL_OK;
}

extern "C" int ddrl_obs_gather(const void* obs_full, int is_f64, int64_t S, int Dfull, const int32_t* table, int Ag, int D,
                               int P, float* out, void* stream) {
    DDRL_REQUIRE(obs_full && table && out && S >= 0 && Dfull >= 1 && Ag >= 1 && D >= 1 && P >= 1 && Ag % P == 0, DDRL_E_BADARG,
                 "obs_gather: null pointer or bad shape (agents must be a multiple of policies)");
    if (S == 0) return DDRL_OK;
    const int nb = (int)std::min<int64_t>(4096, (S * Ag * D + 255) / 256);
    if (is_f64) obs_gather_kernel<double><<<nb, 256, 0, (cudaStream_t)stream>>>((const double*)obs_full, S, Dfull, table, Ag, D, P, out);
    else obs_gather_kernel<float><<<nb, 256, 0, (cudaStream_t)stream>>>((const float*)obs_full, S, Dfull, table, Ag, D, P, out);
    DDRL_CHECK_LAUNCH("obs_gather");
    return DDRL_OK;
}

extern "C" int ddrl_graph_obs_build(const void* obs_full, int is_f64, int64_t S, int Dfull, const int32_t* table, int Ag,
                                    int Dn, const double* mean, const double* stdv, double clip, const double* leg_zw,
                                    int replicate, float* state, int32_t* node_idx, void* stream) {
    DDRL_REQUIRE(S >= 0 && Dfull >= 5 && Ag >= 1 && Dn >= 0, DDRL_E_BADARG,
                 "graph_obs_build: bad shape (the observation must hold the body quaternion in columns 1..4)");
    if (S == 0) return DDRL_OK;      // an empty batch has no buffers to check
    DDRL_REQUIRE(obs_full && table && leg_zw && state, DDRL_E_BADARG, "graph_obs_build: null pointer");
    const int nb = (int)std::min<int64_t>(4096, (S * Ag * (Dn + 4) + 255) / 256);
    cudaStream_t st = (cudaStream_t)stream;
    if (is_f64) graph_obs_build_kernel<double><<<nb, 256, 0, st>>>((const double*)obs_full, S, Dfull, table, Ag, Dn, mean, stdv,
                                                                   clip, leg_zw, replicate, state, node_idx);
    else graph_obs_build_kernel<float><<<nb, 256, 0, st>>>((const float*)obs_full, S, Dfull, table, Ag, Dn, mean, stdv, clip,
                                                           leg_zw, replicate, state, node_idx);
    DDRL_CHECK_LAUNCH("graph_obs_build");
    return DDRL_OK;
}

extern "C" int ddrl_dg_sample(const float* logits, const float* eps, int64_t R, int A, float* action, float* logp,
                              void* stream) {
    DDRL_REQUIRE(logits && eps && action && logp && R >= 0, DDRL_E_BADARG, "dg_sample: null pointer or bad R");
    DDRL_REQUIRE(A >= 1 && A <= DDRL_MAX_ACT, DDRL_E_UNSUPPORTED_SHAPE, "dg_sample: unsupported A=%d", A);
    if (R == 0) return DDRL_OK;
    const int nb = (int)std::min<int64_t>(2048, (R + 255) / 256);
    dg_sample_kernel<<<nb, 256, 0, (cudaStream_t)stream>>>(logits, eps, R, A, action, logp);
    DDRL_CHECK_LAUNCH("dg_sample");
    return DDRL_OK;
}

extern "C" int ddrl_leg_coupling(float* logits, const int32_t* node_id, const float* coupling, int64_t B, int W,
                                 void* stream) {
    DDRL_REQUIRE(logits && node_id && coupling && B >= 0 && W >= 2, DDRL_E_BADARG, "leg_coupling: null pointer or bad shape");
    if (B == 0) return DDRL_OK;
    const int nb = (int)std::min<int64_t>(1024, (B * W + 255) / 256);
    leg_coupling_kernel<<<nb, 256, 0, (cudaStream_t)stream>>>(logits, node_id, coupling, B, W);
    DDRL_CHECK_LAUNCH("leg_coupling");
    return DDRL_OK;
}

extern "C" int ddrl_param_expand(const float* theta_model, const int32_t* map, int P, int NPm, int NPk, float* theta_kernel,
                                 void* stream) {
    DDRL_REQUIRE(theta_model && map && theta_kernel && P >= 1 && NPm >= 1 && NPk >= 1, DDRL_E_BADARG, "param_expand: bad arguments");
    param_expand_kernel<<<dim3((NPk + 255) / 256, P), 256, 0, (cudaStream_t)stream>>>(theta_model, map, NPm, NPk, theta_kernel);
    DDRL_CHECK_LAUNCH("param_expand");
    return DDRL_OK;
}

extern "C" int ddrl_grad_tie(const float* grad_kernel, const int32_t* inv, int P, int NPm, int NPk, float* grad_model, void* stream) {
    DDRL_REQUIRE(grad_kernel && inv && grad_model && P >= 1 && NPm >= 1 && NPk >= 1, DDRL_E_BADARG, "grad_tie: bad arguments");
    grad_tie_kernel<<<dim3((NPm + 255) / 256, P), 256, 0, (cudaStream_t)stream>>>(grad_kernel, inv, NPm, NPk, grad_model);
    DDRL_CHECK_LAUNCH("grad_tie");
    return DDRL_OK;
}

extern "C" int ddrl_leg_coupling_backward(float* dout, const float* logits_pre, const int32_t* node_id, const float* coupling,
                                          int64_t B, int W, float* dcoupling, void* stream) {
    DDRL_REQUIRE(dout && logits_pre && node_id && coupling && dcoupling && B >= 0 && W >= 2, DDRL_E_BADARG,
                 "leg_coupling_backward: null pointer or bad shape");
    leg_coupling_bwd_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(dout, logits_pre, node_id, coupling, B, W, dcoupling);
    DDRL_CHECK_LAUNCH("leg_coupling_backward");
    return DDRL_OK;
}

extern "C" int64_t ddrl_sgd_exchange_words(int NP, int ctas_per_policy) {
    if (NP < 1 || ctas_per_policy < 1) return DDRL_E_BADARG;
    return (int64_t)ctas_per_policy * sgd_slice_len(NP, ctas_per_policy);
}

extern "C" int64_t ddrl_sgd_ll_words(int P, int ctas_per_policy, int D, int A) {
    if (P < 1 || ctas_per_policy < 1 || D < 1 || A < 1) return DDRL_E_BADARG;
    return ll_total_words(P, ctas_per_policy, fc_offsets(D, A).NP);
}

// ---- peer-mapped memory (CUDA IPC) for the in-kernel gradient all-reduce ------------------------------------------------
static_assert(sizeof(cudaIpcMemHandle_t) == 64, "handle64 is a cudaIpcMemHandle_t");

extern "C" int ddrl_peer_alloc(int64_t bytes, void** ptr, void* handle64) {
    DDRL_REQUIRE(bytes > 0 && ptr && handle64, DDRL_E_BADARG, "peer_alloc: bad arguments");
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, (size_t)bytes);
    DDRL_REQUIRE(e == cudaSuccess, DDRL_E_CUDA, "peer_alloc: cudaMalloc(%lld): %s", (long long)bytes, cudaGetErrorString(e));
    e = cudaMemset(p, 0, (size_t)bytes);
    if (e == cudaSuccess) e = cudaIpcGetMemHandle(reinterpret_cast<cudaIpcMemHandle_t*>(handle64), p);
    if (e != cudaSuccess) {
        cudaFree(p);
        set_error("peer_alloc: %s", cudaGetErrorString(e));
        return DDRL_E_CUDA;
    }
    *ptr = p;
    return DDRL_OK;
}

extern "C" int ddrl_peer_open(const void* handle64, void** ptr) {
    DDRL_REQUIRE(handle64 && ptr, DDRL_E_BADARG, "peer_open: bad arguments");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, sizeof(h));
    void* p = nullptr;
    const cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
    DDRL_REQUIRE(e == cudaSuccess, DDRL_E_CUDA, "peer_open: cudaIpcOpenMemHandle: %s", cudaGetErrorString(e));
    *ptr = p;
    return DDRL_OK;
}

extern "C" int ddrl_peer_close(void* ptr) {
    DDRL_REQUIRE(ptr, DDRL_E_BADARG, "peer_close: null pointer");
    const cudaError_t e = cudaIpcCloseMemHandle(ptr);
    DDRL_REQUIRE(e == cudaSuccess, DDRL_E_CUDA, "peer_close: %s", cudaGetErrorString(e));
    return DDRL_OK;
}

extern "C" int ddrl_peer_free(void* ptr) {
    DDRL_REQUIRE(ptr, DDRL_E_BADARG, "peer_free: null pointer");
    const cudaError_t e = cudaFree(ptr);
    DDRL_REQUIRE(e == cudaSuccess, DDRL_E_CUDA, "peer_free: %s", cudaGetErrorString(e));
    return DDRL_OK;
}

extern "C" int ddrl_reward_split(const float* fw_reward, const float* actions, const double* cfrc_ext, const double* contact_table,
                                 int64_t S, int Ag, int A, int NB, double ctrl_cost_weight, double contact_cost_weight, int mode,
                                 float* rewards, void* stream) {
    DDRL_REQUIRE(fw_reward && actions && cfrc_ext && contact_table && rewards && S >= 0, DDRL_E_BADARG, "reward_split: null pointer or bad S");
    DDRL_REQUIRE(Ag >= 1 && Ag <= 8 && A >= 1 && NB >= 1 && NB <= 16 && mode >= 0 && mode <= 3, DDRL_E_UNSUPPORTED_SHAPE,
                 "reward_split: unsupported Ag=%d NB=%d mode=%d (Ag <= 8, NB <= 16, mode 0..3)", Ag, NB, mode);
    if (S == 0) return DDRL_OK;
    reward_split_kernel<<<(unsigned)((S + 127) / 128), 128, 0, (cudaStream_t)stream>>>(fw_reward, actions, cfrc_ext, contact_table, S, Ag,
                                                                                      A, NB, ctrl_cost_weight, contact_cost_weight,
                                                                                      mode, rewards);
    DDRL_CHECK_LAUNCH("reward_split");
    return DDRL_OK;
}

extern "C" int ddrl_concat_actions(const float* actions, const int32_t* action_table, int64_t S, int Ag, int A, int A_full,
                                   float clip_lo, float clip_hi, float* env_actions, void* stream) {
    DDRL_REQUIRE(actions && action_table && env_actions && S >= 0 && Ag >= 1 && A >= 1 && A_full >= Ag * A, DDRL_E_BADARG,
                 "concat_actions: null pointer or bad shape (A_full >= Ag * A)");
    if (S == 0) return DDRL_OK;
    const int64_t n = S * Ag * A;
    concat_actions_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(actions, action_table, S, Ag, A, A_full,
                                                                                        clip_lo, clip_hi, env_actions);
    DDRL_CHECK_LAUNCH("concat_actions");
    return DDRL_OK;
}

// Row-by-row MeanStdFilter streams (RLlib 1.0.1 sampler semantics), as a fixed-order parallel scan of Welford states.
//
// RLlib's sampler (evaluation/sampler.py _process_observations) calls the policy's MeanStdFilter once per observation row,
// unvectorised: push the row into `rs` and `buffer`, then normalise it with the updated state.  Each rollout worker filters
// its own rows, starting from the state the driver gave it; FilterManager.synchronize then folds the workers' buffers into
// the driver copy in worker order.  Here a rollout x[P][R][D], R = T*C rows in (t, c) order, has W streams per policy:
// stream w owns columns [w*C/W, (w+1)*C/W) and visits its rows in (t, c) order.  Three launches, no atomics:
//   1. chunk partials: every FS_CHUNK consecutive rows of a stream, Welford-pushed from an empty state (thread per feature);
//   2. scan: per (policy, stream, feature) one warp; the chunks are split into 32 contiguous groups, lane l folds group l,
//      the group totals are folded in lane order onto the running state (exclusive prefix of every group) and from an
//      empty state (the stream's buffer -> parts), then lane l re-folds its group and leaves every chunk's prefix state;
//   3. re-walk: every chunk is pushed row by row from its prefix state, and every row is normalised with the state after
//      its own push.
// The merge tree is a function of the stream length alone (FS_CHUNK, 32 groups), so the bits do not depend on the launch
// geometry.  All float64 arithmetic uses _rn intrinsics in the reference's operation order (no FMA contraction): a chunk
// walked from the exact sequential state (the first chunk of every stream, walked from the running state itself)
// reproduces RLlib bit for bit; later chunks start from a merged prefix within 1e-12 relative of the sequential one.
#include "common.cuh"

namespace ddrl {

constexpr int FS_CHUNK = 64;     // rows per chunk (tests/test_filter_stream_algorithm.py transcribes the schedule)
constexpr int FS_GROUPS = 32;    // chunk groups of the scan (one lane each)
constexpr int FS_T = 256;

struct WState { double n, M, S; };

// RunningStat.push (ray.rllib.utils.filter): n += 1; the first push sets M = x; else delta = x - M, M += delta / n,
// S += delta * delta * n1 / n
__device__ __forceinline__ void ws_push(WState& s, double x) {
    const double n1 = s.n;
    s.n = __dadd_rn(n1, 1.0);
    if (n1 == 0.0) {
        s.M = x;
    } else {
        const double delta = __dsub_rn(x, s.M);
        s.M = __dadd_rn(s.M, __ddiv_rn(delta, s.n));
        s.S = __dadd_rn(s.S, __ddiv_rn(__dmul_rn(__dmul_rn(delta, delta), n1), s.n));
    }
}

// RunningStat.update: delta = M1 - M2; M = (n1 M1 + n2 M2) / n; S = S1 + S2 + delta^2 n1 n2 / n.  An empty side leaves
// the other unchanged (exact, where the reference's formula may round (n2 M2) / n2).
__device__ __forceinline__ WState ws_merge(const WState& a, const WState& b) {
    if (b.n == 0.0) return a;
    if (a.n == 0.0) return b;
    const double n = __dadd_rn(a.n, b.n);
    const double delta = __dsub_rn(a.M, b.M);
    WState r;
    r.n = n;
    r.M = __ddiv_rn(__dadd_rn(__dmul_rn(a.n, a.M), __dmul_rn(b.n, b.M)), n);
    r.S = __dadd_rn(__dadd_rn(a.S, b.S), __ddiv_rn(__dmul_rn(__dmul_rn(__dmul_rn(delta, delta), a.n), b.n), n));
    return r;
}

template <typename T>
__device__ __forceinline__ double load_x(const T* __restrict__ x, int64_t i) { return (double)__ldg(x + i); }

// thread -> (p, w, chunk k, feature d), d fastest.  Stream row j = k*FS_CHUNK + i -> rollout row (j / Cw)*C + w*Cw + j % Cw
struct ChunkPos { int p, w, d; int64_t k, j0, j1, t, c; };
__device__ __forceinline__ bool chunk_pos(int64_t i, int P, int W, int64_t nch, int D, int64_t L, int64_t Cw, ChunkPos& q) {
    if (i >= (int64_t)P * W * nch * D) return false;
    q.d = (int)(i % D);
    int64_t r = i / D;
    q.k = r % nch;
    r /= nch;
    q.w = (int)(r % W);
    q.p = (int)(r / W);
    q.j0 = q.k * FS_CHUNK;
    q.j1 = min(q.j0 + FS_CHUNK, L);
    q.t = q.j0 / Cw;
    q.c = q.j0 - q.t * Cw;
    return true;
}

template <typename T>
__global__ void __launch_bounds__(FS_T) filter_stream_partial_kernel(const T* __restrict__ x, int P, int64_t C, int W, int D,
                                                                     int64_t L, int64_t nch, double* __restrict__ part) {
    ChunkPos q;
    const int64_t i = (int64_t)blockIdx.x * FS_T + threadIdx.x;
    if (!chunk_pos(i, P, W, nch, D, L, C / W, q)) return;
    const int64_t Cw = C / W, R = L * W;
    const T* xp = x + (int64_t)q.p * R * D + q.d;
    WState s{0.0, 0.0, 0.0};
    int64_t t = q.t, c = q.c;
    for (int64_t j = q.j0; j < q.j1; ++j) {
        ws_push(s, load_x(xp, (t * C + q.w * Cw + c) * D));
        if (++c == Cw) { c = 0; ++t; }
    }
    double* o = part + i * 3;
    o[0] = s.n; o[1] = s.M; o[2] = s.S;
}

__global__ void __launch_bounds__(FS_T) filter_stream_scan_kernel(double* __restrict__ part, int P, int W, int D, int64_t nch,
                                                                  const int64_t* __restrict__ n0, const double* __restrict__ M0,
                                                                  const double* __restrict__ S0, double* __restrict__ parts_out) {
    const int lane = threadIdx.x & 31;
    const int64_t g = ((int64_t)blockIdx.x * FS_T + threadIdx.x) >> 5;     // (p, w, d), d fastest
    if (g >= (int64_t)P * W * D) return;                                    // (whole warps leave together)
    const int d = (int)(g % D), w = (int)((g / D) % W), p = (int)(g / ((int64_t)D * W));
    const int64_t G = (nch + FS_GROUPS - 1) / FS_GROUPS;
    const int64_t k0 = min((int64_t)lane * G, nch), k1 = min(k0 + G, nch);
    double* base = part + ((((int64_t)p * W + w) * nch) * D + d) * 3;
    const int64_t stride = (int64_t)D * 3;
    WState tot{0.0, 0.0, 0.0};
#pragma unroll 4
    for (int64_t k = k0; k < k1; ++k) {
        const double* o = base + k * stride;
        tot = ws_merge(tot, WState{o[0], o[1], o[2]});
    }
    WState pre{(double)n0[p], M0[(int64_t)p * D + d], S0[(int64_t)p * D + d]};
    WState buf{0.0, 0.0, 0.0};
    for (int l = 0; l < FS_GROUPS; ++l) {
        const WState o{__shfl_sync(0xffffffffu, tot.n, l), __shfl_sync(0xffffffffu, tot.M, l), __shfl_sync(0xffffffffu, tot.S, l)};
        if (l < lane) pre = ws_merge(pre, o);
        buf = ws_merge(buf, o);
    }
    if (lane == 0) {
        double* o = parts_out + ((((int64_t)p * W + w) * D) + d) * 3;
        o[0] = buf.n; o[1] = buf.M; o[2] = buf.S;
    }
    for (int64_t k = k0; k < k1; ++k) {      // in place: chunk k's partial is read before its prefix replaces it
        double* o = base + k * stride;
        const WState c{o[0], o[1], o[2]};
        o[0] = pre.n; o[1] = pre.M; o[2] = pre.S;
        pre = ws_merge(pre, c);
    }
}

template <typename T>
__global__ void __launch_bounds__(FS_T) filter_stream_walk_kernel(const T* __restrict__ x, int P, int64_t C, int W, int D,
                                                                  int64_t L, int64_t nch, const double* __restrict__ prefix,
                                                                  double clip, float* __restrict__ out) {
    ChunkPos q;
    const int64_t i = (int64_t)blockIdx.x * FS_T + threadIdx.x;
    if (!chunk_pos(i, P, W, nch, D, L, C / W, q)) return;
    const int64_t Cw = C / W, R = L * W;
    const T* xp = x + (int64_t)q.p * R * D + q.d;
    float* op = out + (int64_t)q.p * R * D + q.d;
    WState s{prefix[i * 3], prefix[i * 3 + 1], prefix[i * 3 + 2]};
    int64_t t = q.t, c = q.c;
    for (int64_t j = q.j0; j < q.j1; ++j) {
        const int64_t row = t * C + q.w * Cw + c;
        const double v = load_x(xp, row * D);
        ws_push(s, v);
        // MeanStdFilter.__call__: (x - mean) / (std + 1e-8), std = sqrt(S / (n - 1)) if n > 1 else sqrt(M^2); clip if set
        const double var = s.n > 1.0 ? __ddiv_rn(s.S, __dsub_rn(s.n, 1.0)) : __dmul_rn(s.M, s.M);
        double y = __ddiv_rn(__dsub_rn(v, s.M), __dadd_rn(__dsqrt_rn(var), 1e-8));
        if (clip > 0.0) y = fmin(fmax(y, -clip), clip);
        op[row * D] = __double2float_rn(y);
        if (++c == Cw) { c = 0; ++t; }
    }
}

}  // namespace ddrl

using namespace ddrl;

static int64_t fs_chunks(int T, int64_t C, int W) { return ((int64_t)T * (C / W) + FS_CHUNK - 1) / FS_CHUNK; }

extern "C" int64_t ddrl_filter_stream_ws_bytes(int P, int T, int64_t C, int W, int D) {
    if (P < 1 || T < 1 || C < 1 || W < 1 || D < 1 || C % W) return DDRL_E_BADARG;
    return (int64_t)P * W * fs_chunks(T, C, W) * D * 3 * (int64_t)sizeof(double);
}

extern "C" int ddrl_filter_stream(const void* x, int x_is_f64, int P, int T, int64_t C, int W, int D, const int64_t* n,
                                  const double* M, const double* S, double clip, float* out, double* parts, void* ws,
                                  void* stream) {
    DDRL_REQUIRE(x && n && M && S && out && parts && ws, DDRL_E_BADARG, "filter_stream: null pointer");
    DDRL_REQUIRE(P >= 1 && T >= 1 && C >= 1 && W >= 1 && D >= 1, DDRL_E_BADARG,
                 "filter_stream: bad shape P=%d T=%d C=%lld W=%d D=%d", P, T, (long long)C, W, D);
    DDRL_REQUIRE(C % W == 0, DDRL_E_BADARG, "filter_stream: C=%lld columns do not split into W=%d equal streams",
                 (long long)C, W);
    DDRL_REQUIRE(D <= DDRL_MAX_OBS, DDRL_E_UNSUPPORTED_SHAPE, "filter_stream: D=%d > %d", D, DDRL_MAX_OBS);
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t L = (int64_t)T * (C / W), nch = fs_chunks(T, C, W);
    const int64_t nt = (int64_t)P * W * nch * D;
    const unsigned blocks = (unsigned)((nt + FS_T - 1) / FS_T);
    const unsigned scan_blocks = (unsigned)(((int64_t)P * W * D * 32 + FS_T - 1) / FS_T);
    double* part = (double*)ws;
    if (x_is_f64) filter_stream_partial_kernel<double><<<blocks, FS_T, 0, st>>>((const double*)x, P, C, W, D, L, nch, part);
    else filter_stream_partial_kernel<float><<<blocks, FS_T, 0, st>>>((const float*)x, P, C, W, D, L, nch, part);
    DDRL_CHECK_LAUNCH("filter_stream_partial");
    filter_stream_scan_kernel<<<scan_blocks, FS_T, 0, st>>>(part, P, W, D, nch, n, M, S, parts);
    DDRL_CHECK_LAUNCH("filter_stream_scan");
    if (x_is_f64) filter_stream_walk_kernel<double><<<blocks, FS_T, 0, st>>>((const double*)x, P, C, W, D, L, nch, part, clip, out);
    else filter_stream_walk_kernel<float><<<blocks, FS_T, 0, st>>>((const float*)x, P, C, W, D, L, nch, part, clip, out);
    DDRL_CHECK_LAUNCH("filter_stream_walk");
    return DDRL_OK;
}

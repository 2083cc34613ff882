// Tensor-core (tcgen05) FCNet training step: packed weight image and shared-memory layout (byte offsets).
#pragma once
#include "common.cuh"

namespace ddrl {

constexpr int TC_ROWS = 128;   // rows per tile = UMMA M
constexpr int TC_NT = 512;     // threads per CTA: thread = (row, 16-column quarter of the 64-wide branch tile)
constexpr int TC_NO = 16;      // head operand width (2A <= 16 outputs; the value head uses column 0)

__host__ __device__ inline int tc_kx(int D) { return (D + 1 + 15) & ~15; }   // >= 1 pad column (holds the constant 1)

// chunked fp16 matrix [rows][cols]: element offset of (r, c), see umma.cuh
__host__ __device__ inline int tc_chunk_off(int rows, int r, int c) { return ((c >> 3) * rows + r) * 8 + (c & 7); }

// Image (== first part of shared memory), per policy.  Branch 0 = policy, 1 = value.  fp16 entries hold 256*w.
//   W1[b][hi|lo] : [64 out c][KX in d] chunked along d    (F1: B operand, K-major)
//   W2[b][hi|lo] : [64 in j][64 out c] chunked along c    (F2: B MN-major;  B4: B K-major)
//   WoT[b][hi|lo]: [16 out o][64 in k] chunked along k    (head: B K-major;  dz2 = dl.Wo^T: B MN-major)
//   f32 block    : b1c[128] b2c[128] bo[16] bvo[4]
struct TcImg {
    int W1[2][2], W2[2][2], WoT[2][2], b1c, b2c, bo, bvo, bytes;
};
__host__ __device__ inline TcImg tc_img(int D, int A) {
    const int KX = tc_kx(D);
    TcImg L;
    int p = 0;
    for (int b = 0; b < 2; ++b)
        for (int h = 0; h < 2; ++h) { L.W1[b][h] = p; p += 64 * KX * 2; }
    for (int b = 0; b < 2; ++b)
        for (int h = 0; h < 2; ++h) { L.W2[b][h] = p; p += 64 * 64 * 2; }
    for (int b = 0; b < 2; ++b)
        for (int h = 0; h < 2; ++h) { L.WoT[b][h] = p; p += TC_NO * 64 * 2; }
    L.b1c = p; p += 128 * 4;
    L.b2c = p; p += 128 * 4;
    L.bo = p;  p += 16 * 4;
    L.bvo = p; p += 16;
    L.bytes = (p + 15) & ~15;
    (void)A;
    return L;
}

struct TcSmem {
    int X[2], H1[2], H2[2], DL[2], xraw, pf, red, bar, total;
};
__host__ __device__ inline TcSmem tc_smem(int D, int A) {
    const int KX = tc_kx(D);
    TcSmem s;
    int p = tc_img(D, A).bytes;
    for (int h = 0; h < 2; ++h) { s.X[h] = p; p += TC_ROWS * KX * 2; }
    for (int h = 0; h < 2; ++h) { s.H1[h] = p; p += TC_ROWS * 64 * 2; }
    for (int h = 0; h < 2; ++h) { s.H2[h] = p; p += TC_ROWS * 64 * 2; }
    for (int h = 0; h < 2; ++h) { s.DL[h] = p; p += TC_ROWS * TC_NO * 2; }
    s.xraw = p;  p += ((TC_ROWS * D * 4) + 15) & ~15;
    s.pf = p;    p += ((TC_ROWS * (3 * A + 4) * 4) + 15) & ~15;
    s.red = p;   p += 4 * 32 * 8;    // [4 warps][<= 32 values] doubles
    s.bar = p;   p += 32;            // mbarrier (8 B) + tmem slot (4 B)
    s.total = p;
    return s;
}


// ---- "ping-pong" kernel (tc2.cu): both branches resident, so the tensor core works on one branch while the CTA runs
// the other branch's epilogue.  H1/H2 of BOTH branches take 128 KB, so two buffers live in space that is dead at the time:
//   * the loss-gradient operand DL[b] sits in the W1 part of the weight image (W1 is only read by F1; a CTA with another
//     tile to go reloads it from L2 behind the backward, and every step reloads the whole image anyway);
//   * the fp32 staging of the observations (xraw) sits in H2[1] (free from B3(1) of one tile to tanh2(1) of the next).
// That fits KX <= 48 (D <= 47) for every A in {1, 2, 4, 8}; below KX = 32 DL (and for A = 8 the old logits) get regions of
// their own.
struct Tc2Smem {
    int X[2], H1[2][2], H2[2][2], DL[2][2], xraw, pf, po, red, bar, nid, cup, total;
    bool dl_in_w1, po_in_w1;
};
// cup: the leg-coupled step (SharedDecentralLegID) also stages the node ids of the tile ([128] int32), the rows' coupling
// table gradients ([128][2]) and the coupling table ([4][2] floats) behind the other regions
__host__ __device__ inline Tc2Smem tc2_smem(int D, int A, bool cup = false) {
    const int KX = tc_kx(D);
    const TcImg I = tc_img(D, A);
    Tc2Smem s;
    int p = I.bytes;
    for (int h = 0; h < 2; ++h) { s.X[h] = p; p += TC_ROWS * KX * 2; }
    for (int b = 0; b < 2; ++b)
        for (int h = 0; h < 2; ++h) { s.H1[b][h] = p; p += TC_ROWS * 64 * 2; }
    for (int b = 0; b < 2; ++b)
        for (int h = 0; h < 2; ++h) { s.H2[b][h] = p; p += TC_ROWS * 64 * 2; }
    const int dl_bytes = 4 * TC_ROWS * TC_NO * 2, w1_bytes = 4 * 64 * KX * 2;
    s.dl_in_w1 = w1_bytes >= dl_bytes;              // KX >= 32
    const int dl0 = s.dl_in_w1 ? I.W1[0][0] : p;
    if (!s.dl_in_w1) p += dl_bytes;
    for (int b = 0; b < 2; ++b)
        for (int h = 0; h < 2; ++h) s.DL[b][h] = dl0 + (2 * b + h) * TC_ROWS * TC_NO * 2;
    s.xraw = s.H2[1][0];                            // 32 KB >= 128 rows x 63 floats
    // staged loss inputs: actions [128][A], old_logits [128][2A], 4 x [128] scalars.  For A = 8 the old logits (8 KB) move
    // into the part of the W1 region that DL leaves free (KX >= 48) and are fetched after F1 has consumed W1.
    s.po_in_w1 = A > 4 && s.dl_in_w1 && w1_bytes >= dl_bytes + TC_ROWS * 2 * A * 4;
    s.pf = p;
    if (s.po_in_w1) { s.po = I.W1[0][0] + dl_bytes; p += ((TC_ROWS * (A + 4) * 4) + 15) & ~15; }
    else            { s.po = p + TC_ROWS * A * 4;   p += ((TC_ROWS * (3 * A + 4) * 4) + 15) & ~15; }
    s.red = p;   p += 8 * 24 * 8;    // [8 loss warps][24] doubles: 5 stat sums, 16 head-bias gradient sums
    s.bar = p;   p += 64;            // 2 mbarriers, tmem slot, 2 gradient scales
    s.nid = s.cup = 0;
    if (cup) { s.nid = p; p += TC_ROWS * 4 * 3; s.cup = p; p += 32; }      // node ids, then the rows' table gradients [128][2]
    s.total = p;
    return s;
}
__host__ __device__ inline bool tc2_eligible(int D, int A) {
    return tc_kx(D) <= 48 && tc2_smem(D, A).total <= 227 * 1024;
}

// Where flat parameter j lives in the image: fp16 pair (byte offsets of hi and lo, f16 = true) or one float.
__host__ __device__ inline void tc_img_pos(const TcImg& L, const FcOffsets& o, int D, int A, int j, bool& f16, int& p0, int& p1) {
    const int A2 = 2 * A;
    f16 = false; p1 = -1;
    auto pair = [&](const int (&buf)[2], int e) { f16 = true; p0 = buf[0] + 2 * e; p1 = buf[1] + 2 * e; };
    if (j < o.b1)       { const int i = j - o.W1;  pair(L.W1[0], tc_chunk_off(64, i & 63, i >> 6)); }
    else if (j < o.Wv1) p0 = L.b1c + (j - o.b1) * 4;
    else if (j < o.bv1) { const int i = j - o.Wv1; pair(L.W1[1], tc_chunk_off(64, i & 63, i >> 6)); }
    else if (j < o.W2)  p0 = L.b1c + (64 + j - o.bv1) * 4;
    else if (j < o.b2)  { const int i = j - o.W2;  pair(L.W2[0], tc_chunk_off(64, i >> 6, i & 63)); }
    else if (j < o.Wv2) p0 = L.b2c + (j - o.b2) * 4;
    else if (j < o.bv2) { const int i = j - o.Wv2; pair(L.W2[1], tc_chunk_off(64, i >> 6, i & 63)); }
    else if (j < o.Wo)  p0 = L.b2c + (64 + j - o.bv2) * 4;
    else if (j < o.bo)  { const int i = j - o.Wo;  const int k = i / A2, q = i - k * A2; pair(L.WoT[0], tc_chunk_off(TC_NO, q, k)); }
    else if (j < o.Wvo) p0 = L.bo + (j - o.bo) * 4;
    else if (j < o.bvo) { const int k = j - o.Wvo; pair(L.WoT[1], tc_chunk_off(TC_NO, 0, k)); }
    else                p0 = L.bvo;
    (void)D;
}

}  // namespace ddrl

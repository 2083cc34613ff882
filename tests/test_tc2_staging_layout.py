"""CPU transcription of the index arithmetic of the ping-pong step kernel's partial-gradient write-out (csrc/tc2.cu, round 2):
the stacked M = 128 weight-gradient accumulators are read out by the four MMA-issue warps into TWO flat-indexed, ROTATED staging
buffers (half 0 over H2, half 1 over the weight image), XOR-swizzled inside the two 64 x 64 blocks, and the copy-out adds the
halves and undoes rotation and swizzle.  The arithmetic below is copied from the kernel (stage_w2 / stage_heads / stage_w1 /
bias_stats / copy_out); the test checks for every shape the ping-pong kernel runs (D <= 47, A in {1, 2, 4, 8}) that
  * both staging buffers fit the memory they live in, and what is staged in "slot 1" (while B4(1) still runs) only touches
    memory that is dead at that time,
  * every flat index of the partial is written exactly once per half (half 1: zeros for the entries without lo-half rows),
  * the three copy-out ranges cover the vector exactly once and deliver flat element j = hi-half value + lo-half value."""
import numpy as np
import pytest

H, TC_ROWS, TC_NO = 64, 128, 16
SHAPES = [(D, A) for A in (1, 2, 4, 8) for D in range(1, 48)]      # every ping-pong shape (tests/test_fcnet_envelope.py)


def fc_offsets(D, A):      # csrc/common.cuh
    names = ["W1", "b1", "Wv1", "bv1", "W2", "b2", "Wv2", "bv2", "Wo", "bo", "Wvo", "bvo"]
    sizes = [D * H, H, D * H, H, H * H, H, H * H, H, H * 2 * A, 2 * A, H, 1]
    o, p = {}, 0
    for n, s in zip(names, sizes):
        o[n] = p
        p += s
    o["NP"] = p
    return o


def tc_kx(D):
    return (D + 1 + 15) & ~15


def image(D):              # csrc/fcnet_tc_layout.cuh tc_img
    KX = tc_kx(D)
    w1, w2, wot = 4 * 64 * KX * 2, 4 * 64 * 64 * 2, 4 * TC_NO * 64 * 2
    f32 = 128 * 4 + 128 * 4 + 16 * 4 + 16
    return {"W1": (0, w1), "W2_0": (w1, w1 + w2 // 2), "W2_1": (w1 + w2 // 2, w1 + w2), "bytes": (w1 + w2 + wot + f32 + 15) & ~15}


@pytest.mark.parametrize("D,A", SHAPES)
def test_staged_partial_round_trip(D, A):
    o = fc_offsets(D, A)
    A2, KX = 2 * A, tc_kx(D)
    NP = o["NP"]
    NPs = (NP + 3) & ~3
    rotn = NPs - o["W2"]
    rot = lambda idx: idx - o["W2"] if idx >= o["W2"] else idx + rotn      # noqa: E731
    img = image(D)
    # -- the buffers fit: half 0 over H2 (both branches, hi | lo: 64 KB), half 1 over the weight image
    assert NPs * 4 <= 4 * TC_ROWS * 64 * 2
    assert NPs * 4 <= img["bytes"]
    assert sorted(rot(i) for i in range(NPs)) == list(range(NPs))
    assert o["W2"] % 64 == 0 and (o["Wv2"] - o["W2"]) % 64 == 0      # block starts are multiples of 16 float4 (XOR stays in the row)

    stage = np.full((2, NPs), np.nan)      # [half][rotated index]
    written = np.zeros((2, NPs), dtype=np.int32)

    def put(half, idx, val):
        assert 0 <= idx < NPs
        stage[half, idx] = val
        written[half, idx] += 1

    # value model: flat element j carries 1000 + j in the hi-half rows and 0.5 * j in the lo-half rows
    hi_v = lambda j: 1000.0 + j      # noqa: E731
    lo_v = lambda j: 0.5 * j         # noqa: E731
    slot1 = np.zeros((2, NPs), dtype=bool)
    for q in range(4):               # MMA warp 16 + q: TMEM lanes 32 q .. 32 q + 31
        for lane in range(32):
            m, half = (32 * q + lane) & 63, int(q >= 2)
            val = (hi_v, lo_v)[half]
            for b in range(2):       # stage_w2(b)
                blk = o["Wv2"] if b else o["W2"]
                rowb, sw = rot(blk) + m * 64, m & 7
                for c16 in range(4):
                    for k in range(4):
                        base = rowb + 4 * ((4 * c16 + k) ^ sw)
                        for e in range(4):
                            col = 4 * (4 * c16 + k) + e
                            put(half, base + e, val(blk + m * 64 + col))
                            if b == 0:
                                slot1[half, base + e] = True
                bb = o["bv2"] if b else o["b2"]
                put(half, rot(bb) + m, val(bb + m))
                if b == 0:
                    slot1[half, rot(bb) + m] = True
            for oo in range(A2):     # stage_heads(0), (1)
                put(half, rot(o["Wo"]) + m * A2 + oo, val(o["Wo"] + m * A2 + oo))
            put(half, rot(o["Wvo"]) + m, val(o["Wvo"] + m))
            for b in range(2):       # stage_w1(b): gW1[d][m] at W1 + 64 d + m, row D = the bias gradient
                blk = o["Wv1"] if b else o["W1"]
                for c8 in range(KX >> 3):
                    i0, jmax = rot(blk) + 512 * c8 + m, D - 8 * c8
                    for j in range(8):
                        if j <= jmax:
                            put(half, i0 + 64 * j, val(blk + 64 * (8 * c8 + j) + m))
    for tid in range(32):            # bias_stats (one warp): head biases, padding floats; zeros in half 1
        if tid < A2:
            put(0, rot(o["bo"]) + tid, hi_v(o["bo"] + tid)); put(1, rot(o["bo"]) + tid, 0.0)
        if tid == A2:
            put(0, rot(o["bvo"]), hi_v(o["bvo"])); put(1, rot(o["bvo"]), 0.0)
        if tid > A2 and NP + (tid - A2 - 1) < NPs:
            put(0, rot(NP) + (tid - A2 - 1), 0.0); put(1, rot(NP) + (tid - A2 - 1), 0.0)
    assert (written == 1).all(), "every element of both staging halves is written exactly once"

    # -- slot 1 (gW2_0, gb2_0, staged while B4(1) is still running) touches only dead memory: the first 32 KB of the H2 region
    #    (H2 of branch 0) in half 0; W1 and the W2 image of branch 0 in half 1
    top = 4 * (int(np.nonzero(slot1.any(axis=0))[0].max()) + 1)
    assert top <= 2 * TC_ROWS * 64 * 2
    assert top <= img["W2_0"][1]

    # -- copy_out: three ranges of flat float4 indices, each element exactly once, rotation and swizzle undone, halves added
    w2a, v2a, n4 = o["W2"] >> 2, o["Wv2"] >> 2, NPs >> 2
    assert o["W2"] % 4 == 0 and o["bo"] % 4 == 0
    out = np.full(NPs, np.nan)
    seen = np.zeros(n4, dtype=np.int32)
    for i0, i1 in ((o["W2"] >> 2, o["bo"] >> 2), (0, o["W2"] >> 2), (o["bo"] >> 2, n4)):
        for i in range(i0, i1):
            r0, r1 = i - w2a, i - v2a
            sw = (r0 >> 4) & 7 if 0 <= r0 < 1024 else (r1 >> 4) & 7 if 0 <= r1 < 1024 else 0
            si = i - w2a if i >= w2a else i + (n4 - w2a)
            so = 4 * (si ^ sw)
            out[4 * i:4 * i + 4] = stage[0, so:so + 4] + stage[1, so:so + 4]
            seen[i] += 1
    assert (seen == 1).all()
    want = np.array([hi_v(j) + lo_v(j) for j in range(NPs)])
    for name in ("bo", "bvo"):                       # no lo-half rows
        n = A2 if name == "bo" else 1
        want[o[name]:o[name] + n] = [hi_v(o[name] + t) for t in range(n)]
    want[NP:] = 0.0
    np.testing.assert_array_equal(out, want)

"""CPU: the pure-host shape functions of the FCNet ABI, tabulated over D = -1..66 x A = 0..9 against the envelope
include/ddrl_b200.h states, and FCNetLearner's construction-time check (the same envelope):
  * FP32 kernels: 1 <= D <= 64, 1 <= A <= 8 (ddrl_fcnet_num_params, ddrl_fcnet_image_floats); the FP32 SGD step
    additionally needs D <= 60 for A = 8 (ddrl_fcnet_train_supported);
  * tensor-core kernels: 1 <= D <= 63, A in {1, 2, 4, 8} (ddrl_fcnet_tc_image_bytes, ddrl_fcnet_train_supported);
  * ping-pong step and tensor-core inference forward: D <= 47 within that (ddrl_tc_pingpong_eligible), none under
    variant 1 (branch-sequential forced)."""
import pytest

from ddrl_b200._lib import DDRLError

UNSUPPORTED = -2          # DDRL_E_UNSUPPORTED_SHAPE
DS, AS = range(-1, 67), range(0, 10)


def _lib():
    from ddrl_b200 import _lib
    return _lib.load()


def fp32_shape(D, A):
    return 1 <= D <= 64 and 1 <= A <= 8


def tc_shape(D, A):
    return 1 <= D <= 63 and A in (1, 2, 4, 8)


def pingpong_shape(D, A):
    return tc_shape(D, A) and D <= 47


def test_num_params_and_fp32_image_size():
    lib = _lib()
    for D in DS:
        for A in AS:
            n, f = lib.ddrl_fcnet_num_params(D, A), lib.ddrl_fcnet_image_floats(D, A)
            if not fp32_shape(D, A):
                assert n == f == UNSUPPORTED, (D, A, n, f)
                continue
            assert n == 128 * D + 130 * A + 8513, (D, A, n)
            # fcnet_layout.cuh weight region: W1c [Dp][128] b1c W2c [64][128] b2c W2Tc [64][132] WhT [20][128] Wo bo Wvo bvo
            Dp = (D + 3) & ~3
            want = Dp * 128 + 128 + 64 * 128 + 128 + 64 * 132 + 20 * 128 + 64 * 2 * A + ((2 * A + 3) & ~3) + 64 + 4
            assert f == want and f % 4 == 0, (D, A, f, want)


def test_tensor_core_image_size():
    lib = _lib()
    for D in DS:
        for A in AS:
            b = lib.ddrl_fcnet_tc_image_bytes(D, A)
            if not tc_shape(D, A):
                assert b == UNSUPPORTED, (D, A, b)
                continue
            KX = (D + 1 + 15) & ~15       # X width: D features + the constant-1 pad column, in 16-column blocks
            # fp16 hi | lo of W1 [64][KX], W2 [64][64], WoT [16][64] per branch, then b1c, b2c [128], bo [16], bvo [4] floats
            want = (4 * 64 * KX * 2 + 4 * 64 * 64 * 2 + 4 * 16 * 64 * 2 + 128 * 4 + 128 * 4 + 16 * 4 + 16 + 15) & ~15
            assert b == want, (D, A, b, want)


def test_pingpong_eligibility_under_each_variant():
    lib = _lib()
    try:
        for variant in (0, 2, 1):
            assert lib.ddrl_tc_set_variant(variant) == 0
            for D in DS:
                for A in AS:
                    want = pingpong_shape(D, A) and variant != 1
                    assert lib.ddrl_tc_pingpong_eligible(D, A) == int(want), (variant, D, A)
    finally:
        lib.ddrl_tc_set_variant(0)
    assert lib.ddrl_tc_set_variant(3) != 0 and lib.ddrl_tc_set_variant(-1) != 0


def test_train_step_envelope():
    """ddrl_fcnet_train_supported derives the FP32 limit from the train kernel's shared-memory layout (fcnet_layout.cuh) and
    the tensor-core one from the image shapes and tc_smem; both must be what the header states."""
    lib = _lib()
    for D in DS:
        for A in AS:
            assert lib.ddrl_fcnet_train_supported(D, A, 0) == int(fp32_shape(D, A) and (A < 8 or D <= 60)), (D, A)
            assert lib.ddrl_fcnet_train_supported(D, A, 1) == int(tc_shape(D, A)), (D, A)


@pytest.mark.parametrize("D,A,mode", [(64, 2, "tc"), (21, 3, "tc"), (19, 9, "tc"), (0, 2, "tc"), (61, 8, "fp32"),
                                      (64, 8, "fp32"), (65, 2, "fp32"), (19, 0, "fp32")])
def test_learner_refuses_at_construction_before_touching_a_device(D, A, mode):
    from ddrl_b200.config import PPOConfig
    from ddrl_b200.learner import FCNetLearner
    with pytest.raises(DDRLError, match=f"D={D}, A={A}"):
        FCNetLearner(2, D, A, PPOConfig(), "cuda", mode=mode)

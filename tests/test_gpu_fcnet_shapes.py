"""GPU parity of the FCNet kernels over the (D, A) envelope their entry points accept, not only at the published shapes.

The published architectures all have D in 19..44 and A in {2, 4, 8}: their tensor-core X operand is 32 or 48 columns wide
(KX = tc_kx(D)) and the ping-pong step runs an instantiation with D as a compile-time constant.  Every other shape runs the
runtime-D ping-pong kernel (fcnet_train_tc2_kernel<A, false, false, 0>) or, for 48 <= D <= 63, only the branch-sequential
kernel, and reaches layout branches the published shapes never take.  Each shape below is chosen for the path it reaches:

  (1, 1), (7, 1)    KX = 16, A = 1: the loss gradient DL gets its own shared-memory region (no W1 restore)
  (15, 8)           KX = 16: the constant-1 pad column is the last X column; A = 8 with DL and old logits outside W1
  (16, 2)           first KX = 32
  (30, 8), (31, 8)  A = 8 at KX = 32: the old logits are staged outside W1 (po_in_w1 == false)
  (32, 1), (46, 4)  first KX = 48 (one W1 gradient block); D = 46
  (47, 2), (47, 8)  the largest ping-pong shapes (KX = 48)
  (48, 4), (63, 1), (63, 8)   KX = 64: branch-sequential tensor-core kernel only, FP32 inference forward
  (64, 2), (21, 3), (12, 7)   FP32 kernels only (D = 64, A outside {1, 2, 4, 8})
  (19, 2)           a published shape as a control of the harness

Weights are the oracle's initialisation, perturbed so that biases, log-std and both heads are non-trivial (logits of order
1); observations come from a synthetic filter (mean, std per feature) with a few outliers beyond the clip.  Bars are the
suite's: 1e-5 of the tensor's scale for forward outputs and loss statistics, 1e-5 (FP32) / 5e-5 (tensor cores) for the
reduced gradient, per variable with the float32 torch twin as in tests/test_gpu_fcnet.py."""
import contextlib

import numpy as np
import pytest
import torch

from tests.test_gpu_fcnet import _cuda_train_step, _oracle_grads, _oracle_iteration
from tests.util import assert_grad_per_variable, scaled_err, t64

pytestmark = pytest.mark.gpu

TOL = 1e-5
TC_GTOL = 5e-5
NEAR_CLIP = 2e-6      # DESIGN.md §2: a row this close to the PPO clip kink may fall on either side in float32
P = 2

SHAPES = [(1, 1), (7, 1), (15, 8), (16, 2), (30, 8), (31, 8), (32, 1), (46, 4), (47, 2), (47, 8), (48, 4), (63, 1), (63, 8),
          (64, 2), (21, 3), (12, 7), (19, 2)]
PINGPONG_SHAPES = [s for s in SHAPES if s[0] <= 47 and s[1] in (1, 2, 4, 8)]


def tc_ok(D, A):
    """Tensor-core SGD step (branch-sequential kernel at least): D <= 63, A in {1, 2, 4, 8}."""
    return 1 <= D <= 63 and A in (1, 2, 4, 8)


def pingpong(D, A):
    """Ping-pong step and tensor-core inference forward: D <= 47, A in {1, 2, 4, 8}."""
    return 1 <= D <= 47 and A in (1, 2, 4, 8)


def fp32_step_ok(D, A):
    """FP32 SGD step: D <= 64, A <= 8, and for A = 8 D <= 60 (shared memory of the train kernel <= 227 KB)."""
    return 1 <= D <= 64 and 1 <= A <= 8 and (A < 8 or D <= 60)


def _oracle():
    import oracle.ddrl_oracle as O
    return O


def _dev(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a))
    return (t.to(dtype) if dtype is not None else t).to("cuda")


@contextlib.contextmanager
def _variant(v):
    from ddrl_b200 import kernels as K
    K.tc_set_variant(v)
    try:
        yield
    finally:
        K.tc_set_variant(0)


def _theta(D, A, seed):
    """[P, NP] float32: oracle init, every variable perturbed; biases ~0.1, heads ~0.15 (logits / value of order 1)."""
    O = _oracle()
    g = torch.Generator().manual_seed(seed)
    th = torch.stack([O.fcnet_init(D, 2 * A, g) for _ in range(P)]).double()
    o = 0
    for name, shp in O.fcnet_shapes(D, 2 * A):
        n = int(np.prod(shp))
        noise = torch.randn(P, n, generator=g, dtype=torch.float64)
        if len(shp) == 1:
            th[:, o:o + n] = 0.1 * noise
        elif name.startswith(("fc_out", "value_out")):
            th[:, o:o + n] = 0.15 * noise
        else:
            th[:, o:o + n] += 0.02 * noise
        o += n
    return th.float().numpy()


def _filter(D, seed):
    rng = np.random.default_rng(seed)
    mean = 2.0 * rng.standard_normal((P, D))
    std = np.exp(rng.uniform(-1.0, 1.0, (P, D)))
    return mean, std


def _raw_obs(mean, std, R, seed):
    """Raw observations ~ N(mean, std^2) with every 37th row of one feature 15 std out (beyond the clip of 10)."""
    rng = np.random.default_rng(seed)
    raw = mean[:, None, :] + std[:, None, :] * rng.standard_normal((P, R, mean.shape[1]))
    raw[:, ::37, (R // 37) % mean.shape[1]] = (mean + 15.0 * std)[:, None, (R // 37) % mean.shape[1]]
    return raw.astype(np.float32)


def _norm(mean, std):
    return np.stack([mean, 1.0 / (std + 1e-8)], axis=1)      # [P, 2, D] float64: the filter's {mean, 1 / (std + eps)}


def _normalise(raw, norm, clip):
    x = ((raw.astype(np.float64) - norm[:, 0][:, None, :]) * norm[:, 1][:, None, :]).astype(np.float32)
    return np.clip(x, -clip, clip) if clip else x


def _batch(D, A, R, seed):
    """A train batch of P policies at shape (D, A): dict of numpy arrays [P, R, ...] (as tests/test_gpu_fcnet._make_batch)."""
    O = _oracle()
    rng = np.random.default_rng(seed + 1)
    theta = _theta(D, A, seed)
    mean, std = _filter(D, seed)
    x = _normalise(_raw_obs(mean, std, R, seed), _norm(mean, std), 10.0)
    logits = np.zeros((P, R, 2 * A), np.float32)
    value = np.zeros((P, R), np.float32)
    for p in range(P):
        lg, v = O.fcnet_forward(t64(theta[p]), t64(x[p]), 2 * A)
        logits[p], value[p] = lg.numpy(), v.numpy()
    eps = rng.standard_normal((P, R, A)).astype(np.float32)
    act = (logits[..., :A] + np.exp(logits[..., A:]) * eps).astype(np.float32)
    old_logits = (logits + 0.05 * rng.standard_normal(logits.shape)).astype(np.float32)
    old_logp = np.stack([O.dg_logp(t64(old_logits[p]), t64(act[p])).numpy() for p in range(P)]).astype(np.float32)
    return {"theta": theta, "obs": x, "D": D, "A": A, "P": P, "actions": act, "old_logits": old_logits, "old_logp": old_logp,
            "vf_preds": (value + 2.0 * rng.standard_normal(value.shape)).astype(np.float32),
            "adv": rng.standard_normal((P, R)).astype(np.float32),
            "vtarg": (value + 1.5 * rng.standard_normal(value.shape)).astype(np.float32), "logits": logits, "value": value,
            "eps": eps}


def _forward_rows(D, A):
    """R = 1; a ragged R; an R whose rows-per-CTA rounding leaves the last CTA of a policy without rows in the tensor-core
    forward; an R > 128 x (CTAs per policy), so that CTAs run several 128-row tiles."""
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    gmax = max(1, sms // P)
    empty = None
    for R in range(128 * gmax + 1, 128 * gmax + 4096):
        G = min(-(-R // 128), gmax)
        rpc = (-(-R // G) + 7) & ~7
        if (G - 1) * rpc >= R:
            empty = R
            break
    assert empty is not None
    return [1, 777, empty, 128 * gmax * 2 + 77]


# ---- forward ------------------------------------------------------------------------------------------------------------
def _check_forward(res, x, theta, eps, A, where):
    """logits, value, action, logp of a forward result against the float64 oracle on the network input x."""
    O = _oracle()
    for p in range(P):
        lg, v = O.fcnet_forward(t64(theta[p]), t64(x[p]), 2 * A)
        assert scaled_err(res["logits"][p].cpu().numpy(), lg.numpy()) < TOL, (*where, p, "logits")
        assert scaled_err(res["value"][p].cpu().numpy(), v.numpy()) < TOL, (*where, p, "value")
        if eps is not None:
            act = O.dg_sample(lg, t64(eps[p]))
            assert scaled_err(res["action"][p].cpu().numpy(), act.numpy()) < TOL, (*where, p, "action")
            assert scaled_err(res["logp"][p].cpu().numpy(), O.dg_logp(lg, act).numpy()) < TOL, (*where, p, "logp")


FWD_PATHS = ("fp32-norm", "fp32", "tc-norm", "tc")


def _forward_checks(D, A, R, seed, corrupt=None, paths=FWD_PATHS):
    """Forward against the oracle on each of `paths`: the FP32 kernel with the filter prologue + clip 10 ("fp32-norm") and on
    already-normalised input ("fp32"), and, where eligible, the tensor-core forward likewise ("tc-norm", "tc").
    corrupt: None, "obs" (column D - 1 of the kernel's input zeroed) or "bias" (fc_1/bias of the kernel's weights off by 1e-3
    relative); the oracle always gets the true values.  A corrupted run skips the checks of the filter prologue's obs_out
    (which reports the corrupted input faithfully), so that what fails is the network's output."""
    from ddrl_b200 import kernels as K
    theta = _theta(D, A, seed)
    mean, std = _filter(D, seed)
    norm = _norm(mean, std)
    raw = _raw_obs(mean, std, R, seed)
    x = _normalise(raw, norm, 10.0)
    eps = np.random.default_rng(seed + 2).standard_normal((P, R, A)).astype(np.float32)
    raw_k, x_k, theta_k = raw.copy(), x.copy(), theta.copy()
    if corrupt == "obs":
        raw_k[:, :, D - 1] = 0.0
        x_k[:, :, D - 1] = 0.0
    elif corrupt == "bias":
        theta_k[:, D * 64:D * 64 + 64] *= 1.0 + 1e-3
    th = _dev(theta_k)
    r32 = None
    if "fp32-norm" in paths or ("tc-norm" in paths and corrupt is None):
        # FP32 kernel, filter prologue + clip
        r32 = K.fcnet_forward(th, _dev(raw_k), A, norm=_dev(norm), clip=10.0, eps=_dev(eps), want_obs_out=True)
        torch.cuda.synchronize()
        if corrupt is None:
            np.testing.assert_allclose(r32["obs_out"].cpu().numpy(), x, rtol=3e-7, atol=1e-7)
    if "fp32-norm" in paths:
        _check_forward(r32, x, theta, eps, A, ("fp32 norm", D, A, R))
    if "fp32" in paths:      # FP32 kernel on already-normalised input, no sampling
        _check_forward(K.fcnet_forward(th, _dev(x_k), A), x, theta, None, A, ("fp32", D, A, R))
    assert K.tc_pingpong_eligible(D, A) == pingpong(D, A)
    if not pingpong(D, A):
        return
    img = K.fcnet_tc_pack(th, D, A)
    if "tc-norm" in paths:
        out = K.fcnet_forward_tc(img, _dev(raw_k), A, norm=_dev(norm), clip=10.0, eps=_dev(eps))
        torch.cuda.synchronize()
        assert int(out["status"]) == 0
        if corrupt is None:
            assert torch.equal(out["obs_out"], r32["obs_out"])
        _check_forward(out, x, theta, eps, A, ("tc norm", D, A, R))
        vb = torch.empty(P, R, dtype=torch.float32, device="cuda")
        K.fcnet_forward_tc(img, _dev(raw_k), A, norm=_dev(norm), clip=10.0, out={"logits": None, "value": vb, "obs_out": None})
        assert torch.equal(vb, out["value"])
    if "tc" in paths:
        _check_forward(K.fcnet_forward_tc(img, _dev(x_k), A), x, theta, None, A, ("tc", D, A, R))


@pytest.mark.parametrize("D,A", SHAPES)
def test_forward_matches_oracle(D, A):
    for R in _forward_rows(D, A):
        _forward_checks(D, A, R, seed=100 * D + A)


# ---- one SGD step -------------------------------------------------------------------------------------------------------
def _step_checks(D, A, tc, corrupt=None):
    """One SGD step (minibatch 1 = rows [500, 1000) of R = 1000, G = 3 CTAs per policy: 168-row CTAs, i.e. two 128-row tiles
    each, the second ragged, and a shorter last CTA) against float64 autograd and the oracle's loss statistics."""
    from ddrl_b200 import kernels as K
    O = _oracle()
    cfg = O.PPOConfig(entropy_coeff=0.01)
    R, MB, G = 1000, 500, 3
    b = _batch(D, A, R, seed=7 * D + A)
    klc = [0.2, 0.3]
    rows = slice(MB, 2 * MB)
    # no row within NEAR_CLIP of the clip kink: the side float32 takes there is not defined by the float64 reference
    for p in range(P):
        lg, _ = O.fcnet_forward(t64(b["theta"][p]), t64(b["obs"][p][rows]), 2 * A)
        ratio = torch.exp(O.dg_logp(lg, t64(b["actions"][p][rows])) - t64(b["old_logp"][p][rows])).numpy()
        assert np.minimum(abs(ratio - 1.0 + cfg.clip_param), abs(ratio - 1.0 - cfg.clip_param)).min() > NEAR_CLIP
    ref, stats = _oracle_grads(b, rows, klc, cfg)
    twin, _ = _oracle_grads(b, rows, klc, cfg, torch.float32)
    if corrupt == "obs":
        b["obs"][:, :, D - 1] = 0.0
    elif corrupt == "bias":
        b["theta"][:, D * 64:D * 64 + 64] *= 1.0 + 1e-3
    grad, ssum = _cuda_train_step(b, MB, 1, G, klc, cfg, tc=tc)
    gtol = TC_GTOL if tc else TOL
    shapes = [shp for _, shp in O.fcnet_shapes(D, 2 * A)]
    for p in range(P):
        assert scaled_err(grad[p], ref[p]) < gtol, (D, A, tc, p)
        assert_grad_per_variable(grad[p], ref[p], twin[p], shapes, gtol, where=(D, A, tc, p))
        s = ssum[p] / MB
        assert abs(s[0] - stats[p]["policy_loss"]) < TOL * max(1.0, abs(stats[p]["policy_loss"]))
        assert abs(s[1] - stats[p]["kl"]) < TOL * max(1.0, abs(stats[p]["kl"]))
        assert abs(s[2] - stats[p]["vf_loss"]) < TOL * abs(stats[p]["vf_loss"])
        assert abs(s[3] - stats[p]["entropy"]) < TOL * max(1.0, abs(stats[p]["entropy"]))
        ev = max(-1.0, 1.0 - (s[7] - s[6] ** 2) / (s[5] - s[4] ** 2))
        assert abs(ev - stats[p]["vf_explained_var"]) < 1e-4


STEP_CASES = [(D, A, tc) for D, A in SHAPES for tc in (False, True, "seq")
              if (fp32_step_ok(D, A) if tc is False else tc_ok(D, A))]


@pytest.mark.parametrize("D,A,tc", STEP_CASES,
                         ids=[f"{D}-{A}-{ {False: 'fp32', True: 'tc', 'seq': 'tc-seq'}[tc]}" for D, A, tc in STEP_CASES])
def test_train_step_gradients_match_float64_autograd(D, A, tc):
    """fp32 = ddrl_ppo_train_step; tc = ddrl_ppo_train_step_tc on its default route (ping-pong where eligible, else the
    branch-sequential kernel); tc-seq = variant 1, the branch-sequential kernel forced."""
    from ddrl_b200 import kernels as K
    with _variant(1 if tc == "seq" else 0):
        assert K.tc_pingpong_eligible(D, A) == (pingpong(D, A) and tc != "seq")
    _step_checks(D, A, tc)


# ---- persistent launch, kept weight images, fused-tail trajectory ---------------------------------------------------------
def _learner_batch(D, A, seed, R=1536):
    b = _batch(D, A, R, seed)
    rng = np.random.default_rng(seed + 5)
    perms = np.stack([np.stack([rng.permutation(4) for _ in range(2)]) for _ in range(P)]).astype(np.int32)
    return b, perms


def _learn(b, perms, **kw):
    from ddrl_b200.config import PPOConfig
    from ddrl_b200.learner import FCNetLearner
    D, A, R = b["D"], b["A"], b["obs"].shape[1]
    L = FCNetLearner(P, D, A, PPOConfig(num_sgd_iter=2, sgd_minibatch_size=R // 4, entropy_coeff=0.01), "cuda",
                     theta=torch.from_numpy(b["theta"]), ctas_per_policy=2, use_graph=False, atomic_reduce=False, **kw)
    stats = L.learn_on_batch(*(_dev(b[k]) for k in ("obs", "actions", "old_logits", "old_logp", "vf_preds", "adv", "vtarg")),
                             _dev(perms), standardize=False)
    torch.cuda.synchronize()
    return L, stats


@pytest.mark.parametrize("D,A", PINGPONG_SHAPES)
def test_persistent_launch_equals_one_step_launches_and_follows_the_oracle(D, A):
    """2 epochs x 4 minibatches of 384 rows on 2 CTAs per policy (192-row CTAs: a full and a ragged 128-row tile each), fused
    tail, fixed-order reduction.  ONE persistent launch of the 8 steps leaves bit-identical state to one launch per step;
    the tensor-core image kept by the tail equals a fresh pack of the updated weights; the trajectory follows the float64
    oracle as closely as the float32 torch twin does."""
    from ddrl_b200 import kernels as K
    O = _oracle()
    b, perms = _learner_batch(D, A, seed=11 * D + A)
    La, sa = _learn(b, perms, mode="tc", persistent=True)
    Lb, sb = _learn(b, perms, mode="tc", persistent=False)
    assert K.tc_pingpong_eligible(D, A)
    assert La._persistent_steps(2) and not Lb._persistent_steps(2)
    for name in ("theta", "m", "v", "beta_pow", "kl_coeff"):
        assert torch.equal(getattr(La, name), getattr(Lb, name)), (D, A, name)
    assert torch.equal(La._bufs["step_stats"], Lb._bufs["step_stats"])
    assert sa == sb
    assert torch.equal(La.tc_img, K.fcnet_tc_pack(La.theta_fc, D, A))
    cfg_o = O.PPOConfig(num_sgd_iter=2, sgd_minibatch_size=b["obs"].shape[1] // 4, entropy_coeff=0.01)
    fwd = lambda th, x: O.fcnet_forward(th, x, 2 * A)      # noqa: E731
    for p in range(P):
        def run(dtype):
            batch = {k: torch.from_numpy(b[src][p]).to(dtype) for k, src in
                     (("obs", "obs"), ("actions", "actions"), ("old_logits", "old_logits"), ("old_logp", "old_logp"),
                      ("vf_preds", "vf_preds"), ("advantages", "adv"), ("value_targets", "vtarg"))}
            t = torch.from_numpy(b["theta"][p]).to(dtype)
            return O.sgd_loop(t, O.AdamState.zeros(t.numel(), dtype, cfg_o), fwd, batch, perms[p], cfg_o.kl_coeff, cfg_o)
        th64, s64 = run(torch.float64)
        th32, _ = run(torch.float32)
        base = b["theta"][p].astype(np.float64)
        upd_o = th64.numpy() - base
        err_dev = scaled_err(La.theta[p].cpu().numpy().astype(np.float64) - base, upd_o)
        err_twin = scaled_err(th32.numpy().astype(np.float64) - base, upd_o)
        assert err_dev < 10.0 * err_twin + 1e-5, (D, A, p, err_dev, err_twin)
        for k in ("total_loss", "policy_loss", "vf_loss", "kl", "entropy", "vf_explained_var"):
            assert abs(sa[p][k] - s64[k]) < 1e-4 * max(1.0, abs(s64[k])), (D, A, p, k, sa[p][k], s64[k])


@pytest.mark.parametrize("D,A,mode", [(1, 1, "fp32"), (15, 8, "fp32"), (47, 8, "fp32"), (64, 2, "fp32"), (12, 7, "fp32"),
                                      (48, 4, "tc"), (63, 1, "tc")])
def test_kept_weight_images_equal_a_fresh_pack(D, A, mode):
    """The fused tail keeps the FP32 image (mode fp32) or the tensor-core image (branch-sequential shapes, one launch per
    step) in step with theta: after 8 steps both equal a fresh pack of the updated weights, bit for bit."""
    from ddrl_b200 import kernels as K
    b, perms = _learner_batch(D, A, seed=13 * D + A, R=768)
    L, _ = _learn(b, perms, mode=mode)
    assert L.fuse_tail and not L._persistent_steps(2)
    assert not torch.equal(L.theta, torch.from_numpy(b["theta"]).cuda())
    if mode == "fp32":
        assert torch.equal(L.img, K.fcnet_pack(L.theta, D, A))
    else:
        assert not K.tc_pingpong_eligible(D, A)
        assert torch.equal(L.tc_img, K.fcnet_tc_pack(L.theta_fc, D, A))


# ---- one whole learner iteration ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("D,A,mode", [(7, 1, "tc"), (30, 8, "tc"), (47, 4, "tc"), (55, 2, "tc"), (64, 3, "fp32")])
def test_full_learner_iteration_matches_oracle(D, A, mode):
    """learn_on_rollout (filter -> forward / sample -> GAE -> standardise -> shuffle -> 2 epochs x 4 minibatches) against
    oracle.fcnet_learner_iteration, with the criteria of tests/test_gpu_fcnet.test_full_learner_iteration_matches_oracle.
    (55, 2) is the tensor-core learner outside the ping-pong envelope: FP32 inference forward and one branch-sequential
    launch per step."""
    from ddrl_b200 import kernels as K
    from ddrl_b200.config import PPOConfig
    from ddrl_b200.learner import FCNetLearner
    O = _oracle()
    T, C, MBS = 16, 32, 128
    R = T * C
    cfgd = dict(num_sgd_iter=2, sgd_minibatch_size=MBS)
    seed = 17 * D + A
    theta0 = _theta(D, A, seed)
    mean, std = _filter(D, seed)
    filt0 = [(1000, mean[p], std[p] ** 2 * 999.0) for p in range(P)]
    rng = np.random.default_rng(seed)
    b = {"D": D, "A": A, "raw": _raw_obs(mean, std, R, seed), "eps": rng.standard_normal((P, R, A)).astype(np.float32)}
    rewards = (0.3 + 0.5 * rng.standard_normal((P, T, C))).astype(np.float32)
    dones = (rng.random((T, C)) < 0.05).astype(np.uint8)
    boot_raw = _raw_obs(mean, std, C, seed + 1)
    perms = np.stack([np.stack([rng.permutation(R // MBS) for _ in range(2)]) for _ in range(P)]).astype(np.int32)
    shuffle = np.stack([rng.permutation(R) for _ in range(P)]).astype(np.int32)

    L = FCNetLearner(P, D, A, PPOConfig(**cfgd), "cuda", theta=torch.from_numpy(theta0), mode=mode)
    _, _, G = L._sgd_setup(R)
    assert K.tc_pingpong_eligible(D, A) == pingpong(D, A)
    assert L._persistent_steps(G) == (mode == "tc" and pingpong(D, A))
    L.filt_n.copy_(torch.tensor([f[0] for f in filt0]))
    L.filt_M.copy_(torch.from_numpy(np.stack([f[1] for f in filt0])))
    L.filt_S.copy_(torch.from_numpy(np.stack([f[2] for f in filt0])))
    stats = L.learn_on_rollout(_dev(b["raw"].reshape(P, T, C, D)), _dev(boot_raw), _dev(rewards), _dev(dones),
                               _dev(b["eps"].reshape(P, T, C, A)), _dev(perms), _dev(shuffle))
    torch.cuda.synchronize()
    cfg_o = O.PPOConfig(**cfgd)
    pols, out = _oracle_iteration(b, theta0, cfg_o, O, torch.float64, perms, shuffle, T, C, dones, boot_raw, rewards, filt0)
    twin, _ = _oracle_iteration(b, theta0, cfg_o, O, torch.float32, perms, shuffle, T, C, dones, boot_raw, rewards, filt0)
    bufs = L._bufs
    for p in range(P):
        assert int(L.filt_n[p]) == pols[p].filt.rs._n == 1000 + R
        np.testing.assert_allclose(L.filt_M[p].cpu().numpy(), pols[p].filt.rs._M, rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(L.filt_S[p].cpu().numpy(), pols[p].filt.rs._S, rtol=1e-11)
        assert scaled_err(bufs["obs"][p].cpu().numpy(), out[p]["obs_norm"]) < 1e-6
        assert scaled_err(bufs["logits"][p].cpu().numpy(), out[p]["logits"].numpy()) < TOL
        assert scaled_err(bufs["value"][p].cpu().numpy(), out[p]["value"].numpy()) < TOL
        assert scaled_err(bufs["act"][p].cpu().numpy(), out[p]["actions"].numpy()) < TOL
        assert scaled_err(bufs["logp"][p].cpu().numpy(), out[p]["logp"].numpy()) < TOL
        assert scaled_err(bufs["vtarg"][p].cpu().numpy(), out[p]["value_targets"].reshape(-1)) < TOL
        assert scaled_err(bufs["adv"][p].cpu().numpy(), out[p]["adv_std"]) < 2e-5
        upd_o = pols[p].theta.numpy() - theta0[p]
        err_dev = scaled_err(L.theta[p].cpu().numpy().astype(np.float64) - theta0[p], upd_o)
        err_twin = scaled_err(twin[p].theta.numpy().astype(np.float64) - theta0[p], upd_o)
        assert err_dev < 10.0 * err_twin + 1e-5, (err_dev, err_twin)
        assert scaled_err(L.theta[p].cpu().numpy(), pols[p].theta.numpy()) < 2e-3
        for k in ("total_loss", "policy_loss", "vf_loss", "kl", "entropy", "vf_explained_var"):
            ref = out[p]["stats"][k]
            assert abs(stats[p][k] - ref) < 1e-4 * max(1.0, abs(ref)), (k, stats[p][k], ref)
        assert abs(L.kl_coeff_host[p] - pols[p].kl_coeff) < 1e-12


# ---- negative controls ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("corrupt", ["obs", "bias"])
@pytest.mark.parametrize("D,A", [(15, 8), (1, 1), (47, 8), (63, 1)])
def test_checks_catch_a_subtly_wrong_kernel_input(D, A, corrupt):
    """The forward and SGD-step checks above must fail when the kernel gets column D - 1 of the observations zeroed (the
    feature next to the constant-1 pad column of the tensor-core X operand) or fc_1/bias off by 1e-3 relative (the bias
    row of W1 in the tensor-core image), while the oracle gets the true values."""
    for path in FWD_PATHS if pingpong(D, A) else FWD_PATHS[:2]:
        with pytest.raises(AssertionError, match="'logits'"):      # the network's output, not a status or obs_out check
            _forward_checks(D, A, 777, seed=100 * D + A, corrupt=corrupt, paths=(path,))
    for tc in ((False, True, "seq") if tc_ok(D, A) else (False,)):
        with pytest.raises(AssertionError):
            _step_checks(D, A, tc, corrupt=corrupt)


# ---- refusals ---------------------------------------------------------------------------------------------------------------
def _step_args(D, A, R=256):
    f32 = torch.float32
    z = lambda *s: torch.zeros(*s, dtype=f32, device="cuda")      # noqa: E731
    NP = 128 * D + 130 * A + 8513
    return dict(obs=z(P, R, D), actions=z(P, R, A), old_logits=z(P, R, 2 * A), old_logp=z(P, R), vf_preds=z(P, R), adv=z(P, R),
                vtarg=z(P, R), gp=z(P, 2, (NP + 3) & ~3), sp=torch.zeros(P, 2, 8, dtype=torch.float64, device="cuda"),
                perm=torch.zeros(P, 1, dtype=torch.int32, device="cuda"), ctr=torch.zeros(1, dtype=torch.int32, device="cuda"),
                klc=z(P), theta=z(P, NP))


def _tc_step(img, D, A):
    from ddrl_b200 import kernels as K
    from ddrl_b200._lib import PPOHyper
    a = _step_args(D, A)
    K.ppo_train_step_tc(img, a["obs"], a["actions"], a["old_logits"], a["old_logp"], a["vf_preds"], a["adv"], a["vtarg"], A, 256,
                        a["perm"], a["ctr"], a["klc"], PPOHyper(0.2, 10.0, 0.5, 0.0, 1 / 256), 2, a["gp"], a["sp"])


def _fp32_step(D, A):
    from ddrl_b200 import kernels as K
    from ddrl_b200._lib import PPOHyper
    a = _step_args(D, A)
    K.ppo_train_step(a["theta"], a["obs"], a["actions"], a["old_logits"], a["old_logp"], a["vf_preds"], a["adv"], a["vtarg"], A,
                     256, a["perm"], a["ctr"], a["klc"], PPOHyper(0.2, 10.0, 0.5, 0.0, 1 / 256), 2, a["gp"], a["sp"])


def test_entry_points_refuse_shapes_outside_their_envelope():
    """On real device buffers of the right sizes: every refusal is an error return before any launch."""
    from ddrl_b200 import kernels as K
    from ddrl_b200._lib import DDRLError
    big = torch.zeros(P, 1 << 17, dtype=torch.uint8, device="cuda")      # larger than any tensor-core image
    theta = lambda D, A: torch.zeros(P, 128 * D + 130 * A + 8513, device="cuda")      # noqa: E731
    obs = lambda D: torch.zeros(P, 64, D, device="cuda")                               # noqa: E731
    # tensor-core entries: D = 64, A outside {1, 2, 4, 8}
    for D, A in [(64, 2), (64, 8), (19, 3), (27, 5), (43, 6), (12, 7)]:
        with pytest.raises(DDRLError, match="unsupported|does not support"):
            K.fcnet_tc_pack(theta(D, A), D, A)
        with pytest.raises(DDRLError, match="unsupported"):
            _tc_step(big, D, A)
        with pytest.raises(DDRLError, match="unsupported"):
            K.fcnet_forward_tc(big, obs(D), A)
        assert not K.tc_pingpong_eligible(D, A)
    # the tensor-core forward and the ping-pong step stop at D = 47; variant 2 (ping-pong forced) refuses D = 48
    for A in (1, 2, 4, 8):
        with pytest.raises(DDRLError, match="unsupported"):
            K.fcnet_forward_tc(K.fcnet_tc_pack(theta(48, A), 48, A), obs(48), A)
        with _variant(2):
            assert not K.tc_pingpong_eligible(48, A) and K.tc_pingpong_eligible(47, A)
            with pytest.raises(DDRLError, match="ping-pong"):
                _tc_step(K.fcnet_tc_pack(theta(48, A), 48, A), 48, A)
    # FP32 SGD step: A = 8 needs D <= 60 (shared memory); D = 60 runs
    for D in (61, 62, 63, 64):
        with pytest.raises(DDRLError, match="shared memory"):
            _fp32_step(D, 8)
    _fp32_step(60, 8)
    torch.cuda.synchronize()

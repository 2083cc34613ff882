"""GPU parity: FCNet grouped forward, fused PPO train step, clip+Adam, SGD loop — CUDA (through the C ABI)
vs the float64 oracle on identical inputs and the reference's checkpoint weights.

Tolerance (north_star): 1e-5 relative in FP32.  "Relative" is taken w.r.t. the tensor's scale for tensors
with entries near zero (scaled_err) and element-wise where the reference value is bounded away from zero."""
import numpy as np
import pytest
import torch

from tests.util import ARCHS, assert_grad_per_variable, ckpt_theta, load_ckpt, scaled_err, synth_obs, t64

pytestmark = pytest.mark.gpu

TOL = 1e-5


def _oracle():
    import oracle.ddrl_oracle as O
    return O


def _norm_from_filter(filt):
    mean = np.stack([M for _, M, _ in filt])
    inv = np.stack([1.0 / (np.sqrt(S / (n - 1)) + 1e-8) for n, _, S in filt])
    return np.stack([mean, inv], axis=1)  # [P,2,D]


def _make_batch(arch, R, seed, dev):
    """Realistic train batch from checkpoint weights: returns dict of numpy arrays [P,R,...]."""
    O = _oracle()
    theta, filt, D, A = ckpt_theta(arch)
    P = theta.shape[0]
    rng = np.random.default_rng(seed)
    raw = synth_obs(filt, R, seed)
    norm = _norm_from_filter(filt)
    x = ((raw.astype(np.float64) - norm[:, 0][:, None, :]) * norm[:, 1][:, None, :]).astype(np.float32)
    out = {"obs": x, "theta": theta, "D": D, "A": A, "P": P, "raw": raw, "norm": norm}
    logits = np.zeros((P, R, 2 * A), np.float32)
    value = np.zeros((P, R), np.float32)
    for p in range(P):
        lg, v = O.fcnet_forward(t64(theta[p]), t64(x[p]), 2 * A)
        logits[p], value[p] = lg.numpy(), v.numpy()
    eps = rng.standard_normal((P, R, A)).astype(np.float32)
    act = (logits[..., :A] + np.exp(logits[..., A:]) * eps).astype(np.float32)
    # "old" policy = slightly perturbed logits so ratio != 1, kl > 0 and both clip branches are exercised
    old_logits = (logits + 0.03 * rng.standard_normal(logits.shape)).astype(np.float32)
    old_logp = np.stack([O.dg_logp(t64(old_logits[p]), t64(act[p])).numpy() for p in range(P)]).astype(np.float32)
    out.update(actions=act, old_logits=old_logits, old_logp=old_logp,
               vf_preds=(value + 12.0 * rng.standard_normal(value.shape)).astype(np.float32),
               adv=rng.standard_normal((P, R)).astype(np.float32),
               vtarg=(value + 8.0 * rng.standard_normal(value.shape)).astype(np.float32),
               logits=logits, value=value, eps=eps)
    return out


def _dev(a, dev, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a))
    if dtype is not None:
        t = t.to(dtype)
    return t.to(dev)


@pytest.mark.parametrize("arch", list(ARCHS))
def test_forward_matches_oracle_on_checkpoint_weights(arch):
    from ddrl_b200 import kernels as K
    O = _oracle()
    dev = "cuda"
    R = 777  # ragged: 12 full tiles + 9 rows
    b = _make_batch(arch, R, 1, dev)
    P, A = b["P"], b["A"]
    res = K.fcnet_forward(_dev(b["theta"], dev), _dev(b["raw"], dev), A, norm=_dev(b["norm"], dev),
                          eps=_dev(b["eps"], dev), want_obs_out=True)
    torch.cuda.synchronize()
    # normalised observation: float64 arithmetic then one rounding to float32 (1/(std+eps) vs division: <= 1 ulp)
    np.testing.assert_allclose(res["obs_out"].cpu().numpy(), b["obs"], rtol=3e-7, atol=1e-7)
    # feed the oracle the exact network input the device used, so the comparison isolates the network
    x_dev = res["obs_out"].cpu().numpy()
    for p in range(P):
        lg, v = O.fcnet_forward(t64(b["theta"][p]), t64(x_dev[p]), 2 * A)
        assert scaled_err(res["logits"][p].cpu().numpy(), lg.numpy()) < TOL
        assert scaled_err(res["value"][p].cpu().numpy(), v.numpy()) < TOL
        act = O.dg_sample(lg, t64(b["eps"][p]))
        assert scaled_err(res["action"][p].cpu().numpy(), act.numpy()) < TOL
        lp = O.dg_logp(lg, act)
        assert scaled_err(res["logp"][p].cpu().numpy(), lp.numpy()) < TOL


@pytest.mark.parametrize("R", [1, 5, 63, 64, 65, 200])
def test_forward_small_and_ragged_batches(R):
    from ddrl_b200 import kernels as K
    O = _oracle()
    b = _make_batch("TwoSides", R, 2, "cuda")
    res = K.fcnet_forward(_dev(b["theta"], "cuda"), _dev(b["obs"], "cuda"), b["A"])
    for p in range(b["P"]):
        lg, v = O.fcnet_forward(t64(b["theta"][p]), t64(b["obs"][p]), 2 * b["A"])
        assert scaled_err(res["logits"][p].cpu().numpy(), lg.numpy()) < TOL
        assert scaled_err(res["value"][p].cpu().numpy(), v.numpy()) < TOL


def _oracle_grads(b, rows, kl_coeff, cfg, dtype=torch.float64):
    """autograd of the mean PPO loss over `rows` for every policy -> grads [P,NP], stats list.
    float64 = ground truth; float32 = the torch twin (what any FP32 implementation can achieve)."""
    O = _oracle()
    P, A = b["P"], b["A"]
    grads, stats = [], []
    t64 = lambda a: torch.from_numpy(np.asarray(a)).to(dtype)
    for p in range(P):
        th = t64(b["theta"][p]).requires_grad_(True)
        lg, v = O.fcnet_forward(th, t64(b["obs"][p][rows]), 2 * A)
        loss, st = O.ppo_loss_from_outputs(lg, v, t64(b["actions"][p][rows]), t64(b["old_logits"][p][rows]),
                                           t64(b["old_logp"][p][rows]), t64(b["vf_preds"][p][rows]),
                                           t64(b["adv"][p][rows]), t64(b["vtarg"][p][rows]), kl_coeff[p], cfg)
        (g,) = torch.autograd.grad(loss, th)
        grads.append(g.numpy())
        stats.append({k: float(x.detach()) for k, x in st.items()})
    return np.stack(grads), stats


def _cuda_train_step(b, MB, mb_index, G, kl_coeff, cfg, dev="cuda", tc=False):
    from ddrl_b200 import kernels as K
    from ddrl_b200._lib import PPOHyper
    P, A = b["P"], b["A"]
    NP = b["theta"].shape[1]
    t = {k: _dev(b[k], dev) for k in ("theta", "obs", "actions", "old_logits", "old_logp", "vf_preds", "adv", "vtarg")}
    gp = torch.full((P, G, K.part_stride(NP)), float("nan"), dtype=torch.float32, device=dev)
    sp = torch.full((P, G, 8), float("nan"), dtype=torch.float64, device=dev)
    grad = torch.empty(P, NP, dtype=torch.float32, device=dev)
    ss = torch.zeros(1, P, 8, dtype=torch.float64, device=dev)
    perm = torch.full((P, 1), mb_index, dtype=torch.int32, device=dev)
    ctr = torch.zeros(1, dtype=torch.int32, device=dev)
    klc = torch.tensor(kl_coeff, dtype=torch.float32, device=dev)
    hyper = PPOHyper(cfg.clip_param, cfg.vf_clip_param, cfg.vf_loss_coeff, cfg.entropy_coeff, 1.0 / MB)
    if tc:
        status = torch.zeros(1, dtype=torch.int32, device=dev)
        img = K.fcnet_tc_pack(t["theta"], b["D"], A)
        K.tc_set_variant(1 if tc == "seq" else 0)      # "seq": force the branch-sequential schedule
        try:
            K.ppo_train_step_tc(img, t["obs"], t["actions"], t["old_logits"], t["old_logp"], t["vf_preds"], t["adv"],
                                t["vtarg"], A, MB, perm, ctr, klc, hyper, G, gp, sp, status)
        finally:
            K.tc_set_variant(0)
        assert int(status) == 0, f"tcgen05 step reported status {int(status)}"
    else:
        K.ppo_train_step(t["theta"], t["obs"], t["actions"], t["old_logits"], t["old_logp"], t["vf_preds"], t["adv"],
                         t["vtarg"], A, MB, perm, ctr, klc, hyper, G, gp, sp)
    K.grad_reduce(gp, sp, P, G, NP, grad, ss, ctr)
    torch.cuda.synchronize()
    return grad.cpu().numpy(), ss.cpu().numpy()[0]


@pytest.mark.parametrize("arch,G", [("FullyDecentral", 1), ("FullyDecentral", 37), ("Centralized", 5),
                                    ("Local", 8), ("Local", 2), ("TwoSides", 3), ("SingleDiagonal", 16),
                                    ("Centralized_TVel", 7), ("FullyDecentral_TVel", 2), ("Local_TVel", 4),
                                    ("TwoSides_TVel", 9)])
@pytest.mark.parametrize("tc", [False, True, "seq"], ids=["fp32", "tcgen05", "tcgen05-seq"])
def test_train_step_gradients_match_float64_autograd(arch, G, tc):
    O = _oracle()
    cfg = O.PPOConfig(entropy_coeff=0.01)  # non-zero so the entropy term is exercised too
    R, MB = 1000, 500                       # minibatch 1 = rows [500, 1000): ragged tiles for most G
    b = _make_batch(arch, R, 3, "cuda")
    klc = [0.2 * 1.5 ** p for p in range(b["P"])]
    grad, ssum = _cuda_train_step(b, MB, 1, G, klc, cfg, tc=tc)
    ref, stats = _oracle_grads(b, slice(MB, 2 * MB), klc, cfg)
    twin, _ = _oracle_grads(b, slice(MB, 2 * MB), klc, cfg, torch.float32)
    # FP32 kernel: 1e-5.  tcgen05 kernel (fp16 hi/lo split, ~22-bit operands): STATED tolerance 5e-5 of the tensor's
    # scale for gradients — the value branch amplifies forward round-off by |v| / |v - R| ~ 10 (the float32 torch twin
    # itself sits at ~5e-6 there); forward outputs and loss statistics stay within 1e-5.
    gtol = 5e-5 if tc else TOL
    z = load_ckpt(arch)
    # checkpoint shape table: [rows, cols], cols = 0 for 1-D variables
    shapes = [(int(r),) if int(c) == 0 else (int(r), int(c)) for r, c in z[[k for k in z.files if k.endswith("/shapes")][0]]]
    for p in range(b["P"]):
        assert scaled_err(grad[p], ref[p]) < gtol, (arch, p)
        assert_grad_per_variable(grad[p], ref[p], twin[p], shapes, gtol, where=(arch, p))
        s = ssum[p] / MB
        assert abs(s[0] - stats[p]["policy_loss"]) < TOL * max(1.0, abs(stats[p]["policy_loss"]))
        assert abs(s[1] - stats[p]["kl"]) < TOL * max(1.0, abs(stats[p]["kl"]))
        assert abs(s[2] - stats[p]["vf_loss"]) < TOL * abs(stats[p]["vf_loss"])
        assert abs(s[3] - stats[p]["entropy"]) < TOL * max(1.0, abs(stats[p]["entropy"]))
        ev = max(-1.0, 1.0 - (s[7] - s[6] ** 2) / (s[5] - s[4] ** 2))
        assert abs(ev - stats[p]["vf_explained_var"]) < 1e-4


def test_train_step_is_bit_reproducible_and_partition_independent_within_tolerance():
    O = _oracle()
    cfg = O.PPOConfig()
    b = _make_batch("FullyDecentral", 512, 4, "cuda")
    klc = [0.2] * 4
    g1, s1 = _cuda_train_step(b, 512, 0, 8, klc, cfg)
    g2, s2 = _cuda_train_step(b, 512, 0, 8, klc, cfg)
    assert np.array_equal(g1, g2) and np.array_equal(s1, s2)      # fixed-order reductions: identical bits
    g3, _ = _cuda_train_step(b, 512, 0, 3, klc, cfg)
    assert scaled_err(g3, g1) < TOL                                  # different CTA split: rounding only


def test_external_gradient_backward_matches_autograd():
    """ModelV2 autograd boundary: dtheta from given dlogits / dvalue."""
    from ddrl_b200 import kernels as K
    O = _oracle()
    b = _make_batch("Local", 300, 5, "cuda")
    P, A = b["P"], b["A"]
    rng = np.random.default_rng(0)
    dl = rng.standard_normal((P, 300, 2 * A)).astype(np.float32)
    dv = rng.standard_normal((P, 300)).astype(np.float32)
    g = K.fcnet_backward(_dev(b["theta"], "cuda"), _dev(b["obs"], "cuda"), _dev(dl, "cuda"), _dev(dv, "cuda"), A)
    for p in range(P):
        th = t64(b["theta"][p]).requires_grad_(True)
        lg, v = O.fcnet_forward(th, t64(b["obs"][p]), 2 * A)
        (ref,) = torch.autograd.grad((lg * t64(dl[p])).sum() + (v * t64(dv[p])).sum(), th)
        assert scaled_err(g[p].cpu().numpy(), ref.numpy()) < TOL


def test_clip_adam_matches_tf1_adam_from_checkpoint_state():
    """TF1 AdamOptimizer semantics, starting from the real m / v / beta powers of a published checkpoint."""
    from ddrl_b200 import kernels as K
    O = _oracle()
    cfg = O.PPOConfig()
    z = load_ckpt("FullyDecentral")
    pids = ARCHS["FullyDecentral"][0]
    theta = np.stack([z[f"{p}/theta"] for p in pids])
    m = np.stack([z[f"{p}/adam_m"] for p in pids])
    v = np.stack([z[f"{p}/adam_v"] for p in pids])
    bp = np.stack([z[f"{p}/beta_powers"] for p in pids])
    # fresh optimizer (beta powers = beta, large correction) and the checkpoint's (saturated) state
    for m0, v0, bp0 in ((np.zeros_like(m), np.zeros_like(v), np.array([[0.9, 0.999]] * 4, np.float32)), (m, v, bp)):
        rng = np.random.default_rng(7)
        dev = "cuda"
        th_d, m_d, v_d, bp_d = (_dev(a.copy(), dev) for a in (theta, m0, v0, bp0))
        sync = torch.zeros(1, dtype=torch.int32, device=dev)
        ctr = torch.zeros(1, dtype=torch.int32, device=dev)
        gn = torch.zeros(4, dtype=torch.float32, device=dev)
        th_o = [torch.from_numpy(theta[p].copy()) for p in range(4)]
        st_o = [O.AdamState(torch.from_numpy(m0[p].copy()), torch.from_numpy(v0[p].copy()), float(bp0[p, 0]),
                            float(bp0[p, 1])) for p in range(4)]
        for step in range(5):
            scale = [0.01, 1.0, 30.0, 1e-4, 3.0][step]   # both sides of the clip threshold 0.5
            g = (scale * rng.standard_normal(theta.shape) / np.sqrt(theta.shape[1])).astype(np.float32)
            K.clip_adam(th_d, m_d, v_d, bp_d, _dev(g, dev), cfg.lr, cfg.beta1, cfg.beta2, cfg.adam_eps, cfg.grad_clip,
                        sync, gn, ctr)
            for p in range(4):
                gc, norm = O.clip_by_global_norm(torch.from_numpy(g[p]), cfg.grad_clip)
                th_o[p] = O.adam_tf1_step(th_o[p], gc, st_o[p], cfg)
                assert abs(float(gn[p]) - float(norm)) < 1e-5 * float(norm)
        torch.cuda.synchronize()
        assert int(ctr) == 5 and int(sync) == 0
        for p in range(4):
            # theta itself agrees to a few float32 ulps (the update is ~1e-3 of |theta|, so ulp-level differences in
            # theta are ~1e-4 of the update: FMA contraction order, not arithmetic); the update agrees to 2e-4
            np.testing.assert_allclose(th_d[p].cpu().numpy(), th_o[p].numpy(), rtol=5e-7, atol=1e-9)
            upd_d = th_d[p].cpu().numpy().astype(np.float64) - theta[p]
            upd_o = th_o[p].numpy().astype(np.float64) - theta[p]
            assert scaled_err(upd_d, upd_o) < 2e-4
            assert scaled_err(m_d[p].cpu().numpy(), st_o[p].m.numpy()) < TOL
            assert scaled_err(v_d[p].cpu().numpy(), st_o[p].v.numpy()) < TOL
            assert abs(float(bp_d[p, 0]) - st_o[p].beta1_power) < 1e-7
            assert abs(float(bp_d[p, 1]) - st_o[p].beta2_power) < 1e-7


def _oracle_iteration(b_np, theta0, cfg, O, dtype, perms, shuffle, T, C, dones, boot_raw, rewards, filt0):
    pols = []
    for p in range(theta0.shape[0]):
        f = O.MeanStdFilter((b_np["D"],), clip=None)
        n, M, S = filt0[p]
        f.rs._n, f.rs._M, f.rs._S = n, M.copy(), S.copy()
        pols.append(O.PolicyState(torch.from_numpy(theta0[p].copy()).to(dtype),
                                  O.AdamState.zeros(theta0.shape[1], dtype, cfg), f, cfg.kl_coeff))
    raw = b_np["raw"].reshape(theta0.shape[0], T, C, -1)
    eps = b_np["eps"].reshape(theta0.shape[0], T, C, -1)
    out = O.fcnet_learner_iteration(pols, raw, boot_raw, rewards, dones, eps, shuffle, perms, 2 * b_np["A"], cfg, dtype)
    return pols, out


@pytest.mark.parametrize("mode", ["fp32", "tc", "tc-fixed", "fp32-3k", "tc-3k", "tc-1step", "tc-cluster", "tc-multitile",
                                  "tc-multitile-fixed", "tc-ll", "tc-llmt"])
@pytest.mark.parametrize("arch,use_graph,use_shuffle", [("FullyDecentral", True, True), ("TwoSides", False, False),
                                                        ("Centralized", True, False)])
def test_full_learner_iteration_matches_oracle(arch, use_graph, use_shuffle, mode):
    """filter -> forward/sample -> GAE -> standardise -> 2 epochs x 4 minibatches of clip+Adam -> KL update.
    "-3k" = the three-kernel SGD step (train, grad_reduce, clip_adam) instead of the fused tail; "-1step" = one launch
    per optimizer step instead of one persistent launch per epoch.  "-ll" = the opt-in LL tail (partial gradients as
    self-validating words pulled by TMA bulk copies, csrc/sgd_tail.cuh) at 32 CTAs per policy; "-llmt" = the same with two
    128-row tiles per CTA (24 CTAs per policy x 136 rows).  "-fixed" = the fixed-order reduction of the per-CTA partial
    gradients (atomic_reduce=False) instead of the default accumulation vector at L2 (red.global.add)."""
    fixed = mode.endswith("-fixed")
    if fixed:
        mode = mode[:-len("-fixed")]
    fuse = not mode.endswith("-3k")
    llmt = mode.endswith("-llmt")
    ll = mode.endswith("-ll") or llmt
    persistent = not mode.endswith("-1step")      # "tc": one persistent launch per epoch where the kernel allows it
    cluster = mode.endswith("-cluster")           # thread-block clusters pre-reduce the partial gradients over DSMEM
    multitile = mode.endswith("-multitile")       # 2 CTAs per policy x 256 rows: two 128-row tiles per CTA, persistent launch
    mode = mode.split("-")[0]
    from ddrl_b200.config import PPOConfig
    from ddrl_b200.learner import FCNetLearner
    O = _oracle()
    T, C = (16, 128) if multitile else (16, 408) if llmt else (16, 32)
    R = T * C
    MBS = 512 if multitile else 3264 if llmt else 128
    cfgd = dict(num_sgd_iter=2, sgd_minibatch_size=MBS)
    cfg_o = O.PPOConfig(**cfgd)
    cfg = PPOConfig(**cfgd)
    b = _make_batch(arch, R, 6, "cuda")
    P, D, A = b["P"], b["D"], b["A"]
    theta0, filt0, _, _ = ckpt_theta(arch)
    # shrink the filter history so this batch visibly moves the statistics
    filt0 = [(1000, M, S * (999.0 / (n - 1))) for n, M, S in filt0]
    rng = np.random.default_rng(11)
    rewards = (0.3 + 0.5 * rng.standard_normal((P, T, C))).astype(np.float32)
    dones = (rng.random((T, C)) < 0.05).astype(np.uint8)
    boot_raw = synth_obs(ckpt_theta(arch)[1], C, 99)
    nb = R // MBS
    perms = np.stack([np.stack([rng.permutation(nb) for _ in range(2)]) for _ in range(P)]).astype(np.int32)
    shuffle = np.stack([rng.permutation(R) for _ in range(P)]).astype(np.int32) if use_shuffle else None

    L = FCNetLearner(P, D, A, cfg, "cuda", theta=torch.from_numpy(theta0), use_graph=use_graph, mode=mode, fuse_tail=fuse,
                     persistent=persistent, ctas_per_policy=8 if cluster else 2 if multitile else 24 if llmt else None,
                     ll_tail=ll, atomic_reduce=not fixed)
    if cluster:
        from ddrl_b200 import kernels as K
        K.tc_set_cluster(-1)
    L.filt_n.copy_(torch.tensor([f[0] for f in filt0]))
    L.filt_M.copy_(torch.from_numpy(np.stack([f[1] for f in filt0])))
    L.filt_S.copy_(torch.from_numpy(np.stack([f[2] for f in filt0])))
    dev = "cuda"
    stats = L.learn_on_rollout(_dev(b["raw"].reshape(P, T, C, D), dev), _dev(boot_raw, dev), _dev(rewards, dev),
                               _dev(dones, dev), _dev(b["eps"].reshape(P, T, C, A), dev), _dev(perms, dev),
                               _dev(shuffle, dev) if use_shuffle else None)
    torch.cuda.synchronize()
    if cluster:
        used = K.tc_last_cluster()
        K.tc_set_cluster(1)
        if K.tc_pingpong_eligible(D, A):
            assert used in (2, 4, 8), f"cluster launch expected, got cluster size {used}"

    pols, out = _oracle_iteration(b, theta0, cfg_o, O, torch.float64, perms, shuffle, T, C, dones, boot_raw, rewards, filt0)
    twin, _ = _oracle_iteration(b, theta0, cfg_o, O, torch.float32, perms, shuffle, T, C, dones, boot_raw, rewards, filt0)
    bufs = L._bufs
    for p in range(P):
        # filter state: count exact, mean / M2 to 1e-12 of the sequential float64 order
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
        # weights after 8 optimizer steps.  Adam normalises every element by its own gradient magnitude, so elements
        # whose gradient is at FP32 round-off level move differently in ANY float32 implementation; the meaningful
        # statement is "no further from the float64 trajectory than the float32 torch twin of the oracle is".
        upd_o = pols[p].theta.numpy() - theta0[p]
        err_dev = scaled_err(L.theta[p].cpu().numpy().astype(np.float64) - theta0[p], upd_o)
        err_twin = scaled_err(twin[p].theta.numpy().astype(np.float64) - theta0[p], upd_o)
        assert err_dev < 10.0 * err_twin + 1e-5, (err_dev, err_twin)
        assert scaled_err(L.theta[p].cpu().numpy(), pols[p].theta.numpy()) < 2e-3
        for k in ("total_loss", "policy_loss", "vf_loss", "kl", "entropy", "vf_explained_var"):
            ref = out[p]["stats"][k]
            assert abs(stats[p][k] - ref) < 1e-4 * max(1.0, abs(ref)), (k, stats[p][k], ref)
        assert abs(L.kl_coeff_host[p] - pols[p].kl_coeff) < 1e-12


def test_packed_weight_image_path_equals_flat_path():
    """The SGD loop feeds the kernels a packed shared-memory image of the weights (kept in step by clip_adam);
    forward, train step and the Adam-maintained image must agree bit for bit with the flat-theta path."""
    from ddrl_b200 import kernels as K
    O = _oracle()
    cfg = O.PPOConfig()
    for arch in ("FullyDecentral", "Centralized_TVel", "TwoSides"):
        b = _make_batch(arch, 300, 9, "cuda")
        P, A, D = b["P"], b["A"], b["D"]
        th = _dev(b["theta"], "cuda")
        img = K.fcnet_pack(th, D, A)
        r1 = K.fcnet_forward(th, _dev(b["obs"], "cuda"), A)
        r2 = K.fcnet_forward(th, _dev(b["obs"], "cuda"), A, img=img)
        assert torch.equal(r1["logits"], r2["logits"]) and torch.equal(r1["value"], r2["value"])
        # Adam-maintained image == re-packed image of the updated theta
        NP = th.shape[1]
        m, v = torch.zeros_like(th), torch.zeros_like(th)
        bp = torch.tensor([[0.9, 0.999]] * P, device="cuda")
        g = torch.randn(P, NP, device="cuda") * 0.01
        sync = torch.zeros(1, dtype=torch.int32, device="cuda")
        K.clip_adam(th, m, v, bp, g, cfg.lr, cfg.beta1, cfg.beta2, cfg.adam_eps, cfg.grad_clip, sync, img=img, img_D=D, img_A=A)
        assert torch.equal(img, K.fcnet_pack(th, D, A))


@pytest.mark.parametrize("arch", ["FullyDecentral", "Local", "TwoSides", "Centralized", "SingleDiagonal", "FullyDecentral_TVel"])
@pytest.mark.parametrize("R", [1, 100, 128, 700, 6528, 20011])      # 20011: several 128-row tiles per CTA, ragged last tile;
# 6528: the rows-per-CTA rounding leaves the last CTA of a policy WITHOUT rows (it wrote through a null partial-gradient
# pointer before round 2)
def test_tensor_core_inference_forward_matches_oracle(arch, R):
    """ddrl_fcnet_forward_tc: filter normalise -> logits / value -> DiagGaussian sample + logp, on checkpoint weights with
    the checkpoint's filter; 1e-5 of the tensor's scale vs the float64 oracle; obs_out identical to the FP32 kernel's."""
    from ddrl_b200 import kernels as K
    O = _oracle()
    theta, filt, D, A = ckpt_theta(arch)
    P = theta.shape[0]
    rng = np.random.default_rng(R)
    raw = synth_obs(filt, R, 7)
    eps = rng.standard_normal((P, R, A)).astype(np.float32)
    norm = np.stack([np.stack([M, 1.0 / (np.sqrt(S / (n - 1)) + 1e-8)]) for n, M, S in filt])
    th = _dev(theta, "cuda")
    img = K.fcnet_tc_pack(th, D, A)
    out = K.fcnet_forward_tc(img, _dev(raw, "cuda"), A, norm=_dev(norm, "cuda"), eps=_dev(eps, "cuda"))
    ref32 = K.fcnet_forward(th, _dev(raw, "cuda"), A, norm=_dev(norm, "cuda"), eps=_dev(eps, "cuda"), want_obs_out=True)
    torch.cuda.synchronize()
    assert int(out["status"]) == 0
    assert torch.equal(out["obs_out"], ref32["obs_out"])
    for p in range(P):
        x = ((raw[p].astype(np.float64) - norm[p, 0]) * norm[p, 1]).astype(np.float32)
        lg, v = O.fcnet_forward(t64(theta[p]), t64(x), 2 * A)
        act = O.dg_sample(lg, t64(eps[p]))
        lp = O.dg_logp(lg, act)
        assert scaled_err(out["logits"][p].cpu().numpy(), lg.numpy()) < TOL
        assert scaled_err(out["value"][p].cpu().numpy(), v.numpy()) < TOL
        assert scaled_err(out["action"][p].cpu().numpy(), act.numpy()) < TOL
        assert scaled_err(out["logp"][p].cpu().numpy(), lp.numpy()) < TOL
    # value-only call (bootstrap): no eps, no logits
    vb = torch.empty(P, R, dtype=torch.float32, device="cuda")
    K.fcnet_forward_tc(img, _dev(raw, "cuda"), A, norm=_dev(norm, "cuda"), out={"logits": None, "value": vb, "obs_out": None})
    assert torch.equal(vb, out["value"])


@pytest.mark.parametrize("atomic", [False, True])
def test_graph_replayed_iterations_are_bit_identical_to_eager_ones(atomic):
    """use_graph=True replays the preparation phase (filter, inference, GAE, shuffle) from a CUDA graph keyed by the input
    buffers; three consecutive iterations must leave exactly the state the eager learner reaches — bit for bit with the
    fixed-order reduction of the partial gradients (atomic_reduce=False); with the default accumulation vector at L2
    (red.global.add: the order of the float additions is not fixed) to round-off."""
    from ddrl_b200.config import PPOConfig
    from ddrl_b200.learner import FCNetLearner
    arch, T, C = "FullyDecentral", 16, 32
    R = T * C
    b = _make_batch(arch, R, 9, "cuda")
    P, D, A = b["P"], b["D"], b["A"]
    theta0, filt0, _, _ = ckpt_theta(arch)
    rng = np.random.default_rng(3)
    rewards = _dev((0.3 + 0.5 * rng.standard_normal((P, T, C))).astype(np.float32), "cuda")
    dones = _dev((rng.random((T, C)) < 0.05).astype(np.uint8), "cuda")
    boot = _dev(synth_obs(filt0, C, 5), "cuda")
    raw = _dev(b["raw"].reshape(P, T, C, D), "cuda")
    eps = _dev(b["eps"].reshape(P, T, C, A), "cuda")
    perms = _dev(np.stack([np.stack([rng.permutation(R // 128) for _ in range(2)]) for _ in range(P)]).astype(np.int32), "cuda")
    shuffle = _dev(np.stack([rng.permutation(R) for _ in range(P)]).astype(np.int32), "cuda")
    out = []
    for graph in (True, False):
        L = FCNetLearner(P, D, A, PPOConfig(num_sgd_iter=2, sgd_minibatch_size=128), "cuda", theta=torch.from_numpy(theta0),
                         use_graph=graph, atomic_reduce=atomic)
        stats = [L.learn_on_rollout(raw, boot, rewards, dones, eps, perms, shuffle) for _ in range(3)]
        torch.cuda.synchronize()
        if graph:
            assert L._prep_graphs is not None and len(L._prep_graphs) == 1, getattr(L, "graph_error", None)
        out.append((L.theta.clone(), L.m.clone(), L.v.clone(), L.filt_M.clone(), L.filt_n.clone(), stats))
    if atomic:
        assert torch.equal(out[0][3], out[1][3]) and torch.equal(out[0][4], out[1][4])      # filter state: no atomics involved
        # 24 Adam steps apart, element by element: Adam turns last-bit gradient differences into O(lr) differences only for
        # elements whose gradient is at round-off level, so compare against the size of the update
        upd = (out[1][0] - torch.from_numpy(theta0).cuda()).abs().max().item()
        assert (out[0][0] - out[1][0]).abs().max().item() < 2e-2 * upd
        return
    for x, y in zip(out[0][:5], out[1][:5]):
        assert torch.equal(x, y)
    assert out[0][5] == out[1][5]


@pytest.mark.parametrize("mode", ["fp32", "tc"])
@pytest.mark.parametrize("vf_share,free_std", [(True, False), (False, True), (True, True)])
def test_learner_trains_the_optional_layouts_like_the_oracle(vf_share, free_std, mode):
    """`vf_share_layers` / `free_log_std` (models/fcnet_glorot_uniform_init.py:30-36,85-113) in the fused learner: the
    kernels run on the index-select of the model's variables, tied gradients are added, clip + Adam act on the model
    variables.  2 epochs x 4 minibatches on postprocessed columns against the oracle's float64 trajectory of the SAME layout."""
    from ddrl_b200.config import PPOConfig
    from ddrl_b200.learner import FCNetLearner
    O = _oracle()
    P, D, A, R, E, NB = 2, 19, 2, 512, 2, 4
    cfgd = dict(num_sgd_iter=E, sgd_minibatch_size=R // NB, entropy_coeff=0.01)
    cfg, cfg_o = PPOConfig(**cfgd), O.PPOConfig(**cfgd)
    g = torch.Generator().manual_seed(17)
    th0 = torch.stack([O.fcnet_init(D, 2 * A, g, vf_share_layers=vf_share, free_log_std=free_std) for _ in range(P)])
    th0 = th0 + 0.05 * torch.randn(th0.shape, generator=g)          # non-zero biases / log_std, larger heads
    rng = np.random.default_rng(5)
    obs = rng.standard_normal((P, R, D)).astype(np.float32)
    old_logits = (0.3 * rng.standard_normal((P, R, 2 * A))).astype(np.float32)
    actions = (old_logits[..., :A] + np.exp(old_logits[..., A:]) * rng.standard_normal((P, R, A))).astype(np.float32)
    old_logp = np.stack([O.dg_logp(torch.from_numpy(old_logits[p]), torch.from_numpy(actions[p])).numpy() for p in range(P)]).astype(np.float32)
    vf_preds = rng.standard_normal((P, R)).astype(np.float32)
    adv = rng.standard_normal((P, R)).astype(np.float32)
    vtarg = (vf_preds + 2.0 * rng.standard_normal((P, R))).astype(np.float32)
    perms = np.stack([np.stack([rng.permutation(NB) for _ in range(E)]) for _ in range(P)]).astype(np.int32)
    L = FCNetLearner(P, D, A, cfg, "cuda", theta=th0.float(), mode=mode, vf_share_layers=vf_share, free_log_std=free_std)
    stats = L.learn_on_batch(_dev(obs, "cuda"), _dev(actions, "cuda"), _dev(old_logits, "cuda"), _dev(old_logp, "cuda"),
                             _dev(vf_preds, "cuda"), _dev(adv, "cuda"), _dev(vtarg, "cuda"), _dev(perms, "cuda"), standardize=False)
    torch.cuda.synchronize()
    fwd = lambda th, x: O.fcnet_forward(th, x, 2 * A, vf_share_layers=vf_share, free_log_std=free_std)
    for p in range(P):
        def run(dtype):
            batch = {"obs": torch.from_numpy(obs[p]).to(dtype), "actions": torch.from_numpy(actions[p]).to(dtype),
                     "old_logits": torch.from_numpy(old_logits[p]).to(dtype), "old_logp": torch.from_numpy(old_logp[p]).to(dtype),
                     "vf_preds": torch.from_numpy(vf_preds[p]).to(dtype), "advantages": torch.from_numpy(adv[p]).to(dtype),
                     "value_targets": torch.from_numpy(vtarg[p]).to(dtype)}
            t = th0[p].float().to(dtype)
            return O.sgd_loop(t, O.AdamState.zeros(t.numel(), dtype, cfg_o), fwd, batch, perms[p], cfg_o.kl_coeff, cfg_o)
        th64, s64 = run(torch.float64)
        th32, _ = run(torch.float32)
        base = th0[p].float().numpy().astype(np.float64)
        upd_o = th64.numpy() - base
        err_dev = scaled_err(L.theta_model[p].cpu().numpy().astype(np.float64) - base, upd_o)
        err_twin = scaled_err(th32.numpy().astype(np.float64) - base, upd_o)
        assert err_dev < 10.0 * err_twin + 1e-5, (err_dev, err_twin)
        assert scaled_err(L.theta_model[p].cpu().numpy(), th64.numpy()) < 2e-3
        # the kernel-layout vector is the index-select of the trained variables (tied copies identical)
        sel = torch.cat([L.theta_model[p], L.theta_model.new_zeros(1)])[L.layout_map.long().clamp(max=L.NPm)]
        assert torch.equal(L.theta[p], sel)
        for k in ("total_loss", "policy_loss", "vf_loss", "kl", "entropy", "vf_explained_var"):
            assert abs(stats[p][k] - s64[k]) < 1e-4 * max(1.0, abs(s64[k])), (k, stats[p][k], s64[k])

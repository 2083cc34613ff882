"""GPU: the leg-coupled SGD steps of SharedDecentralLegID (model "cup" = FCNet + LegCoupling,
models/coupling_net_glorot_uniform_init.py:11-30,135) — ddrl_ppo_train_step_tc_coupled (ping-pong tcgen05 kernel) and
ddrl_ppo_train_step_coupled (FP32 kernel).

  * teacher-forced per-step gradient of all NP + 8 parameters (FCNet variables, then leg_coupling [4, 2]) against float64
    autograd of the oracle's coupled loss, per variable with the table as its own variable, plus the step statistics;
  * with the table == 1 the per-CTA partials and stat partials are bit-identical to the uncoupled kernels';
  * a node-id column shifted by one leg fails the check on the table and on the output layer (negative control);
  * wrong shapes / options and out-of-range node ids fail loudly."""
import numpy as np
import pytest
import torch

from tests.util import assert_grad_per_variable, ckpt_theta, scaled_err, synth_obs, t64

pytestmark = pytest.mark.gpu

TABLE = np.array([[0.7, -1.3], [-0.4, 0.9], [1.6, -0.2], [-1.1, 0.5]], np.float32)   # non-initial: a wrong multiply shows
TOL = 1e-5


def _oracle():
    import oracle.ddrl_oracle as O
    return O


def _shapes(D, A):
    O = _oracle()
    return [tuple(s) for _, s in O.fcnet_shapes(D, 2 * A)] + [(4, 2)]


def _batch(R, seed, table=TABLE, D=19, drop_node=None):
    """Batch of one shared coupled policy on checkpoint FCNet weights: node ids cycle FL, HL, HR, FR (env-major columns);
    the stored old logits are COUPLED logits (perturbed, so that ratio != 1 and both clip branches occur)."""
    O = _oracle()
    theta_all, filt, D0, A = ckpt_theta("FullyDecentral_TVel" if D == 20 else "FullyDecentral")
    assert D0 == D and A == 2
    rng = np.random.default_rng(seed)
    raw = synth_obs(filt[:1], R, seed)[0]
    n, M, S = filt[0]
    x = ((raw.astype(np.float64) - M) / (np.sqrt(S / (n - 1)) + 1e-8)).astype(np.float32)
    node = (np.arange(R) % 4).astype(np.int32)
    rng.shuffle(node)
    if drop_node is not None:
        node[node == drop_node] = (drop_node + 1) % 4
    theta = np.concatenate([theta_all[0], table.reshape(-1)]).astype(np.float32)
    NP = theta_all.shape[1]
    lg, v = O.fcnet_forward(t64(theta[:NP]), t64(x), 2 * A)
    lg = O.leg_coupling(lg, torch.from_numpy(node), t64(table)).numpy().astype(np.float32)
    v = v.numpy().astype(np.float32)
    eps = rng.standard_normal((R, A)).astype(np.float32)
    act = (lg[:, :A] + np.exp(lg[:, A:]) * eps).astype(np.float32)
    old_logits = (lg + 0.03 * rng.standard_normal(lg.shape)).astype(np.float32)
    old_logp = O.dg_logp(t64(old_logits), t64(act)).numpy().astype(np.float32)
    return {"theta": theta, "NP": NP, "D": D, "A": A, "obs": x, "node": node, "actions": act, "old_logits": old_logits,
            "old_logp": old_logp, "vf_preds": (v + 12.0 * rng.standard_normal(R)).astype(np.float32),
            "adv": rng.standard_normal(R).astype(np.float32),
            "vtarg": (v + 8.0 * rng.standard_normal(R)).astype(np.float32)}


def _ref_grad(b, rows, klc, cfg, dtype=torch.float64, node=None):
    """autograd of the mean coupled PPO loss over `rows` w.r.t. the whole [NP + 8] vector -> (grad, stats)."""
    O = _oracle()
    NP, A = b["NP"], b["A"]
    t = lambda a: torch.from_numpy(np.asarray(a)).to(dtype)
    th = t(b["theta"]).requires_grad_(True)
    lg, v = O.fcnet_forward(th[:NP], t(b["obs"][rows]), 2 * A)
    nd = torch.from_numpy(np.asarray(b["node"] if node is None else node)[rows])
    lg = O.leg_coupling(lg, nd, th[NP:].reshape(4, 2))
    loss, st = O.ppo_loss_from_outputs(lg, v, t(b["actions"][rows]), t(b["old_logits"][rows]), t(b["old_logp"][rows]),
                                       t(b["vf_preds"][rows]), t(b["adv"][rows]), t(b["vtarg"][rows]), klc, cfg)
    (g,) = torch.autograd.grad(loss, th)
    return g.numpy(), {k: float(x.detach()) for k, x in st.items()}


def _step(b, MB, mb_index, G, klc, cfg, kind, node=None, coupled=True, dev="cuda"):
    """One step (nsteps = 1) with the fused tail: -> dict(grad = reduced gradient, stats = step stat sums, grad_part,
    stat_part, status).  coupled=False runs the uncoupled kernel of the same kind on theta[:NP]."""
    from ddrl_b200 import kernels as K
    from ddrl_b200._lib import PPOHyper
    NP, A, D = b["NP"], b["A"], b["D"]
    NPk = NP + 8 if coupled else NP
    f32 = torch.float32
    d = lambda a, dt=None: torch.from_numpy(np.ascontiguousarray(a)).to(dev) if dt is None else \
        torch.from_numpy(np.ascontiguousarray(a)).to(dt).to(dev)
    theta = d(b["theta"][:NPk][None])
    obs = d(b["obs"][None])
    cols = {k: d(b[k][None]) for k in ("actions", "old_logits", "old_logp", "vf_preds", "adv", "vtarg")}
    nid = d((b["node"] if node is None else node)[None].astype(np.int32))
    m, v = torch.zeros_like(theta), torch.zeros_like(theta)
    grad = torch.zeros_like(theta)
    beta_pow = torch.tensor([[cfg.beta1, cfg.beta2]], dtype=f32, device=dev)
    bar = torch.zeros(8, dtype=torch.int32, device=dev)
    sq = torch.zeros(1, G, 32, dtype=f32, device=dev)
    gp = torch.full((1, G, K.part_stride(NPk)), float("nan"), dtype=f32, device=dev)
    sp = torch.full((1, G, 8), float("nan"), dtype=torch.float64, device=dev)
    ss = torch.zeros(1, 1, 8, dtype=torch.float64, device=dev)
    perm = torch.full((1, 1), mb_index, dtype=torch.int32, device=dev)
    ctr = torch.zeros(1, dtype=torch.int32, device=dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    kl = torch.tensor([klc], dtype=f32, device=dev)
    hyper = PPOHyper(cfg.clip_param, cfg.vf_clip_param, cfg.vf_loss_coeff, cfg.entropy_coeff, 1.0 / MB)
    if kind == "tc":
        img = K.fcnet_tc_pack(theta[:, :NP].contiguous(), D, A)
        tail = K.make_sgd_tail(theta, m, v, beta_pow, grad, bar, sq, cfg.lr, cfg.beta1, cfg.beta2, cfg.adam_eps, cfg.grad_clip,
                               tc_img=img, step_stats=ss, step_ctr=ctr, status=status)
        if coupled:
            K.ppo_train_step_tc_coupled(img, theta, nid, obs, *cols.values(), A, MB, perm, ctr, kl, hyper, G, gp, sp, status, tail)
        else:
            K.ppo_train_step_tc(img, obs, *cols.values(), A, MB, perm, ctr, kl, hyper, G, gp, sp, status, tail=tail)
    else:
        img = K.fcnet_pack(theta[:, :NP].contiguous(), D, A)
        tail = K.make_sgd_tail(theta, m, v, beta_pow, grad, bar, sq, cfg.lr, cfg.beta1, cfg.beta2, cfg.adam_eps, cfg.grad_clip,
                               img=img, step_stats=ss, step_ctr=ctr, status=status)
        if coupled:
            K.ppo_train_step_coupled(theta, img, nid, obs, *cols.values(), A, MB, perm, ctr, kl, hyper, G, gp, sp, tail)
        else:
            K.ppo_train_step(theta, obs, *cols.values(), A, MB, perm, ctr, kl, hyper, G, gp, sp, img=img, tail=tail)
    torch.cuda.synchronize()
    return {"grad": grad[0].cpu().numpy(), "stats": ss[0, 0].cpu().numpy(), "grad_part": gp[0].cpu().numpy(),
            "stat_part": sp[0].cpu().numpy(), "status": int(status), "theta": theta[0].cpu().numpy()}


# (R, MB, minibatch, G, dropped node): ragged tiles; G * rows-per-CTA > MB leaves CTAs without rows; node 2 absent
CASES = [(1000, 500, 1, 5, None), (600, 300, 1, 37, None), (512, 512, 0, 3, 2)]


@pytest.mark.parametrize("R,MB,mbi,G,drop", CASES, ids=["ragged", "empty-ctas", "missing-node"])
@pytest.mark.parametrize("kind", ["tc", "fp32"])
def test_coupled_step_gradient_matches_float64_autograd(kind, R, MB, mbi, G, drop):
    O = _oracle()
    cfg = O.PPOConfig(entropy_coeff=0.01)
    b = _batch(R, 11, drop_node=drop)
    klc = 0.3
    out = _step(b, MB, mbi, G, klc, cfg, kind)
    assert out["status"] == 0
    rows = slice(mbi * MB, mbi * MB + MB)
    ref, st = _ref_grad(b, rows, klc, cfg)
    twin, _ = _ref_grad(b, rows, klc, cfg, torch.float32)
    gtol = 5e-5 if kind == "tc" else TOL
    assert out["grad"].shape == ref.shape == (b["NP"] + 8,)
    assert scaled_err(out["grad"], ref) < gtol
    assert_grad_per_variable(out["grad"], ref, twin, _shapes(b["D"], b["A"]), gtol, where=(kind, R, G))
    if drop is not None:      # a node without rows in the minibatch: its table-gradient row is exactly 0
        assert np.all(out["grad"][b["NP"] + 2 * drop: b["NP"] + 2 * drop + 2] == 0.0)
    s = out["stats"] / MB
    assert abs(s[0] - st["policy_loss"]) < TOL * max(1.0, abs(st["policy_loss"]))
    assert abs(s[1] - st["kl"]) < TOL * max(1.0, abs(st["kl"]))
    assert abs(s[2] - st["vf_loss"]) < TOL * abs(st["vf_loss"])
    assert abs(s[3] - st["entropy"]) < TOL * max(1.0, abs(st["entropy"]))


@pytest.mark.parametrize("kind", ["tc", "fp32"])
def test_coupled_step_negative_control_shifted_node_ids(kind):
    """A kernel that ignored node_id (or read the wrong leg's row) must fail the check of the test above: feed the ids
    shifted by one leg and require that the table and the output-layer kernel are flagged."""
    O = _oracle()
    cfg = O.PPOConfig(entropy_coeff=0.01)
    b = _batch(1000, 11)
    out = _step(b, 500, 1, 5, 0.3, cfg, kind, node=((b["node"] + 1) % 4).astype(np.int32))
    ref, _ = _ref_grad(b, slice(500, 1000), 0.3, cfg)
    twin, _ = _ref_grad(b, slice(500, 1000), 0.3, cfg, torch.float32)
    gtol = 5e-5 if kind == "tc" else TOL
    NP = b["NP"]
    shapes = _shapes(b["D"], b["A"])
    o_wo = sum(int(np.prod(s)) for s in shapes[:8])        # fc_out/kernel: the policy output layer
    with pytest.raises(AssertionError):
        assert_grad_per_variable(out["grad"][NP:], ref[NP:], twin[NP:], [(4, 2)], gtol)
    with pytest.raises(AssertionError):
        assert_grad_per_variable(out["grad"][o_wo:o_wo + 64 * 4], ref[o_wo:o_wo + 64 * 4], twin[o_wo:o_wo + 64 * 4],
                                 [(64, 4)], gtol)


@pytest.mark.parametrize("kind", ["tc", "fp32"])
def test_table_of_ones_is_bit_identical_to_the_uncoupled_step(kind):
    """Multiplying by 1 is exact: with the table == 1 the coupled kernel's per-CTA partials (first NP entries) and stat
    partials equal the uncoupled kernel's bit for bit (fixed-order reduction, same G, one step)."""
    O = _oracle()
    cfg = O.PPOConfig(entropy_coeff=0.01)
    b = _batch(1000, 5, table=np.ones((4, 2), np.float32))
    cp = _step(b, 500, 1, 7, 0.3, cfg, kind)
    un = _step(b, 500, 1, 7, 0.3, cfg, kind, coupled=False)
    NP = b["NP"]
    assert np.array_equal(cp["grad_part"][:, :NP].view(np.uint32), un["grad_part"][:, :NP].view(np.uint32))
    assert np.array_equal(cp["stat_part"].view(np.uint64), un["stat_part"].view(np.uint64))
    assert np.array_equal(cp["stats"].view(np.uint64), un["stats"].view(np.uint64))


@pytest.mark.parametrize("kind", ["tc", "fp32"])
def test_out_of_range_node_id_sets_the_status_bit(kind):
    from ddrl_b200 import kernels as K
    O = _oracle()
    cfg = O.PPOConfig()
    b = _batch(256, 2)
    node = b["node"].copy()
    node[[3, 100]] = [4, -1]
    out = _step(b, 256, 0, 2, 0.2, cfg, kind, node=node)
    assert out["status"] & K.STATUS_BAD_NODE
    assert np.all(np.isfinite(out["theta"]))


def test_coupled_steps_reject_unsupported_arguments():
    from ddrl_b200 import kernels as K
    from ddrl_b200._lib import DDRLError, PPOHyper
    O = _oracle()
    cfg = O.PPOConfig()
    dev = "cuda"
    b = _batch(256, 2)
    NP = b["NP"]
    f32 = torch.float32

    def args(P=1, A=2, D=19):
        NPk = K.fcnet_num_params(D, A) + 8
        th = torch.zeros(P, NPk, dtype=f32, device=dev)
        z = lambda *s: torch.zeros(*s, dtype=f32, device=dev)
        cols = [z(P, 256, A), z(P, 256, 2 * A), z(P, 256), z(P, 256), z(P, 256), z(P, 256)]
        tail = K.make_sgd_tail(th, torch.zeros_like(th), torch.zeros_like(th), z(P, 2), torch.zeros_like(th),
                               torch.zeros(4 * P + 4, dtype=torch.int32, device=dev), z(P, 2, 32), 1e-4, 0.9, 0.999, 1e-8, 0.5)
        return th, torch.zeros(P, 256, dtype=torch.int32, device=dev), z(P, 256, D), cols, tail

    hyper = PPOHyper(cfg.clip_param, cfg.vf_clip_param, cfg.vf_loss_coeff, cfg.entropy_coeff, 1.0 / 256)
    kl = torch.zeros(4, dtype=f32, device=dev)
    ctr = torch.zeros(1, dtype=torch.int32, device=dev)
    st = torch.zeros(1, dtype=torch.int32, device=dev)

    def tc(P=1, A=2, D=19, tail_on=True, theta_other=False):
        th, nid, obs, cols, tail = args(P, A, D)
        img = K.fcnet_tc_pack(th[:, :K.fcnet_num_params(D, A)].contiguous(), D, A)
        gp = torch.zeros(P, 2, K.part_stride(th.shape[1]), dtype=f32, device=dev)
        sp = torch.zeros(P, 2, 8, dtype=torch.float64, device=dev)
        K.ppo_train_step_tc_coupled(img, th.clone() if theta_other else th, nid, obs, *cols, A, 256, None, ctr, kl, hyper, 2,
                                    gp, sp, st, tail if tail_on else None)

    def fp(P=1, A=2, D=19, tail_on=True):
        th, nid, obs, cols, tail = args(P, A, D)
        img = K.fcnet_pack(th[:, :K.fcnet_num_params(D, A)].contiguous(), D, A)
        gp = torch.zeros(P, 2, K.part_stride(th.shape[1]), dtype=f32, device=dev)
        sp = torch.zeros(P, 2, 8, dtype=torch.float64, device=dev)
        K.ppo_train_step_coupled(th, img, nid, obs, *cols, A, 256, None, ctr, kl, hyper, 2, gp, sp, tail if tail_on else None)

    for fn in (tc, fp):
        with pytest.raises(DDRLError, match="A = 2"):
            fn(A=4, D=27)
        with pytest.raises(DDRLError, match="P = 1"):
            fn(P=2)
        with pytest.raises(DDRLError, match="fused tail is required"):
            fn(tail_on=False)
    with pytest.raises(DDRLError, match="tail->theta"):
        tc(theta_other=True)
    with pytest.raises(DDRLError, match="SharedDecentralLegID"):
        tc(D=27)
    K.tc_set_cluster(2)
    try:
        with pytest.raises(DDRLError, match="clusters"):
            tc()
    finally:
        K.tc_set_cluster(1)
    K.tc_set_variant(1)
    try:
        with pytest.raises(DDRLError, match="ping-pong"):
            tc()
    finally:
        K.tc_set_variant(0)
    torch.cuda.synchronize()
    assert NP == K.fcnet_num_params(19, 2)


# ---- the learner: FCNetLearner(leg_coupling=True) and PPOPolicyGroup on SharedDecentralLegID ---------------------------

def _rollout(T, N, seed):
    """N envs x 4 legs (env-major columns), D = 19, A = 2."""
    rng = np.random.default_rng(seed)
    C = 4 * N
    raw = (rng.standard_normal((T, C, 19)) * 2.0 + 0.5).astype(np.float32)
    boot = (rng.standard_normal((C, 19)) * 2.0 + 0.5).astype(np.float32)
    rew = (0.3 + 0.5 * rng.standard_normal((T, C))).astype(np.float32)
    denv = (rng.random((T, N)) < 0.05).astype(np.uint8)
    eps = rng.standard_normal((T, C, 2)).astype(np.float32)
    return raw, boot, rew, denv, eps


def _learner(theta0, kind, cfg, **kw):
    from ddrl_b200.learner import FCNetLearner
    mode = "fp32" if kind == "fp32" else "tc"
    return FCNetLearner(1, 19, 2, cfg, "cuda", theta=theta0[None], mode=mode, leg_coupling=True,
                        atomic_reduce=(kind == "tc-atomic"), **kw)


def _run_iters(L, iters, T, N, E, MB, seed):
    rng = np.random.default_rng(seed + 100)
    R = T * 4 * N
    to = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    out = []
    for it in range(iters):
        raw, boot, rew, denv, eps = _rollout(T, N, seed + it)
        sh = rng.permutation(R).astype(np.int32)
        perms = np.stack([rng.permutation(R // MB) for _ in range(E)]).astype(np.int32)
        st = L.learn_on_rollout(to(raw[None]), to(boot[None]), to(rew[None]), to(denv), to(eps[None]), to(perms[None]),
                                shuffle=to(sh[None]), cols_per_env=4)
        out.append((raw, boot, rew, np.repeat(denv, 4, axis=1), eps, sh, perms, st))
    torch.cuda.synchronize()
    return out


def _theta0():
    O = _oracle()
    th = O.fcnet_init(19, 4, torch.Generator().manual_seed(7))
    return torch.cat([th, torch.from_numpy(TABLE.reshape(-1))])


@pytest.mark.parametrize("kind", ["tc-fixed", "tc-atomic", "fp32"])
def test_learner_iterations_match_the_float64_coupled_trajectory(kind):
    """3 iterations x E * nb steps (tc: one persistent launch per iteration) against tests/coupling_oracle.py in float64;
    the device's distance to it must stay within 10x the float32 twin's distance (plus 1e-4 of the update)."""
    from tests.coupling_oracle import coupled_learner_iteration
    O = _oracle()
    T, N, E, MB = 16, 8, 2, 128
    cfg = PPOConfig_(E, MB)
    th0 = _theta0()
    L = _learner(th0, kind, cfg)
    runs = _run_iters(L, 3, T, N, E, MB, seed=3)
    cfg_o = O.PPOConfig(num_sgd_iter=E, sgd_minibatch_size=MB)
    traj = {}
    for dt in (torch.float64, torch.float32):
        ps = O.PolicyState(th0.to(dt).clone(), O.AdamState.zeros(th0.numel(), dt, cfg_o), O.MeanStdFilter((19,), clip=None),
                           cfg_o.kl_coeff)
        for raw, boot, rew, dones, eps, sh, perms, _ in runs:
            res = coupled_learner_iteration(ps, raw, boot, rew, dones, eps, sh, perms, cfg_o, dt)
        traj[dt] = (ps, res)
    ref, twin = traj[torch.float64][0], traj[torch.float32][0]
    upd = float((ref.theta - th0.double()).abs().max())
    for name, dev, r, t in (("theta", L.theta[0], ref.theta, twin.theta), ("m", L.m[0], ref.adam.m, twin.adam.m),
                            ("v", L.v[0], ref.adam.v, twin.adam.v)):
        d = dev.detach().cpu().double()
        e_dev = float((d - r).abs().max())
        e_twin = float((t.double() - r).abs().max())
        scale = upd if name == "theta" else float(r.abs().max())
        assert e_dev <= 10 * e_twin + 1e-4 * scale, (kind, name, e_dev, e_twin, scale)
        if name == "theta":      # the table itself, as its own variable
            e_dev_t = float((d[-8:] - r[-8:]).abs().max())
            e_twin_t = float((t.double()[-8:] - r[-8:]).abs().max())
            assert e_dev_t <= 10 * e_twin_t + 1e-4 * upd, (kind, "leg_coupling", e_dev_t, e_twin_t)
            assert float((d[-8:] - th0.double()[-8:]).abs().max()) > 0      # the table trains
    bp = L.beta_pow[0].cpu().double()
    assert abs(float(bp[0]) - ref.adam.beta1_power) < 1e-6 and abs(float(bp[1]) - ref.adam.beta2_power) < 1e-6
    assert float(L.kl_coeff_host[0]) == ref.kl_coeff
    st_dev, st_ref = runs[-1][-1][0], traj[torch.float64][1]["stats"]
    for k in ("policy_loss", "vf_loss", "kl", "entropy"):
        assert abs(st_dev[k] - st_ref[k]) < 1e-3 * max(1.0, abs(st_ref[k])), (kind, k, st_dev[k], st_ref[k])


def PPOConfig_(E, MB):
    from ddrl_b200.config import PPOConfig
    return PPOConfig(num_sgd_iter=E, sgd_minibatch_size=MB)


def test_persistent_launch_is_bit_identical_to_one_launch_per_step():
    th0 = _theta0()
    cfg = PPOConfig_(2, 128)
    A_ = _learner(th0, "tc-fixed", cfg)
    B_ = _learner(th0, "tc-fixed", cfg, persistent=False, use_graph=False)
    _run_iters(A_, 2, 16, 8, 2, 128, seed=5)
    _run_iters(B_, 2, 16, 8, 2, 128, seed=5)
    for a, b in ((A_.theta, B_.theta), (A_.m, B_.m), (A_.v, B_.v)):
        assert torch.equal(a, b)


@pytest.mark.parametrize("kind", ["tc-fixed", "fp32"])
def test_learn_on_batch_is_bit_identical_to_the_sgd_phase_of_learn_on_rollout(kind):
    th0 = _theta0()
    cfg = PPOConfig_(2, 128)
    A_ = _learner(th0, kind, cfg)
    runs = _run_iters(A_, 1, 16, 8, 2, 128, seed=9)
    b = A_._bufs
    sh, perms = runs[0][5], runs[0][6]
    B_ = _learner(th0, kind, cfg)
    to = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    B_.learn_on_batch(b["obs"].clone(), b["act"].clone(), b["logits"].clone(), b["logp"].clone(), b["value"].clone(),
                      b["adv"].clone(), b["vtarg"].clone(), to(perms[None]), to(sh[None]), standardize=False,
                      node_idx=b["node"].clone())
    torch.cuda.synchronize()
    assert torch.equal(A_.theta, B_.theta) and torch.equal(A_.m, B_.m) and torch.equal(A_.v, B_.v)


def test_learner_rejects_unsupported_options_and_bad_node_ids():
    from ddrl_b200._lib import DDRLError
    from ddrl_b200.learner import FCNetLearner
    from ddrl_b200 import checkpoint
    th0 = _theta0()
    cfg = PPOConfig_(1, 128)
    for kw in ({"fuse_tail": False}, {"ll_tail": True}, {"vf_share_layers": True}):
        with pytest.raises(DDRLError):
            FCNetLearner(1, 19, 2, cfg, "cuda", theta=th0[None], leg_coupling=True, **kw)
    with pytest.raises(DDRLError):
        FCNetLearner(2, 19, 2, cfg, "cuda", leg_coupling=True)
    with pytest.raises(DDRLError):
        FCNetLearner(1, 27, 4, cfg, "cuda", leg_coupling=True)
    L = _learner(th0, "tc-fixed", cfg)
    assert torch.equal(FCNetLearner(1, 19, 2, cfg, "cuda", leg_coupling=True).theta[0, -8:].cpu(),
                       torch.tensor([1.0, 1.0, -1.0, -1.0, -1.0, -1.0, 1.0, 1.0]))
    with pytest.raises(ValueError, match="leg-coupled"):
        checkpoint.from_learner(L, ["policy_legs"])
    raw, boot, rew, denv, eps = _rollout(8, 8, 1)
    to = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    with pytest.raises(DDRLError, match="cols_per_env"):
        L.learn_on_rollout(to(raw[None]), to(boot[None]), to(rew[None]), to(denv), to(eps[None]),
                           to(np.zeros((1, 1, 2), np.int32)), cols_per_env=1)
    R = 256
    node = torch.zeros(1, R, dtype=torch.int32, device="cuda")
    node[0, 5] = 7
    z = lambda *s: torch.zeros(*s, dtype=torch.float32, device="cuda")
    with pytest.raises(DDRLError, match="node id"):
        L.learn_on_batch(z(1, R, 19), z(1, R, 2), z(1, R, 4), z(1, R), z(1, R), torch.randn(1, R, device="cuda"), z(1, R),
                         to(np.zeros((1, 1, 2), np.int32)), standardize=False, node_idx=node)


def test_policy_group_on_shared_decentral_leg_id():
    from ddrl_b200.rllib_policy import BatchError, PPOPolicyGroup
    O = _oracle()
    g = PPOPolicyGroup("QuantrupedMultiEnv_SharedDecentralLegID", {"sgd_minibatch_size": 128, "num_sgd_iter": 2}, seed=0)
    pid = g.policy_names[0]
    w = g.get_weights()
    assert w[pid][f"{pid}/leg_coupling"].tolist() == [[1.0, 1.0], [-1.0, -1.0], [-1.0, -1.0], [1.0, 1.0]]
    w[pid][f"{pid}/leg_coupling"] = TABLE.copy()
    g.set_weights(w)
    w2 = g.get_weights()
    assert all(np.array_equal(w2[pid][k], w[pid][k]) for k in w[pid])
    rng = np.random.default_rng(2)
    B = 300
    obs = rng.standard_normal((B, 19)).astype(np.float32)
    node = rng.integers(0, 4, B)
    out = g.compute_actions({pid: (node, obs)}, explore=False)[pid]
    th = torch.from_numpy(g.learner.theta[0].cpu().numpy()).double()
    NP = th.numel() - 8
    lg, v = O.fcnet_forward(th[:NP], torch.from_numpy(obs).double(), 4)
    lg = O.leg_coupling(lg, torch.from_numpy(node), th[NP:].reshape(4, 2))
    assert scaled_err(out[2]["action_dist_inputs"], lg.numpy()) < TOL
    assert scaled_err(out[2]["vf_preds"], v.numpy()) < TOL
    assert scaled_err(out[0], lg[:, :2].numpy()) < TOL
    assert scaled_err(out[2]["action_logp"], O.dg_logp(lg, lg[:, :2]).numpy()) < TOL
    with pytest.raises(BatchError):
        g.compute_actions({pid: (np.full(B, 4), obs)})
    # one learn_on_batch with a ragged tail (300 rows -> 2 whole minibatches of 128), against the oracle on the kept rows
    act = out[0] + 0.1 * rng.standard_normal((B, 2)).astype(np.float32)
    batch = {"obs": obs, "node_idx": node, "actions": act, "action_dist_inputs": out[2]["action_dist_inputs"],
             "action_logp": O.dg_logp(lg, torch.from_numpy(act).double()).numpy().astype(np.float32),
             "vf_preds": out[2]["vf_preds"], "advantages": rng.standard_normal(B).astype(np.float32),
             "value_targets": (out[2]["vf_preds"] + rng.standard_normal(B)).astype(np.float32)}
    state = np.random.RandomState(0)
    state.set_state(g.rng.get_state())
    with pytest.raises(BatchError):
        g.learn_on_batch({pid: {k: v for k, v in batch.items() if k != "node_idx"}})
    stats = g.learn_on_batch({pid: batch})[pid]["learner_stats"]
    shuffle = state.permutation(B)
    perms = np.stack([state.permutation(2) for _ in range(2)])
    from tests.coupling_oracle import coupled_forward
    cfg_o = O.PPOConfig(num_sgd_iter=2, sgd_minibatch_size=128)
    adv = batch["advantages"].astype(np.float64)
    adv_std = (adv - adv.mean()) / max(1e-4, adv.std())
    keep = shuffle[:256]
    t = lambda a: torch.from_numpy(np.asarray(a, dtype=np.float64)[keep])
    ob = {"obs": torch.cat([t(node)[:, None], t(obs)], 1), "actions": t(act), "old_logits": t(batch["action_dist_inputs"]),
          "old_logp": t(batch["action_logp"]), "vf_preds": t(batch["vf_preds"]), "advantages": t(adv_std),
          "value_targets": t(batch["value_targets"])}
    st = O.AdamState.zeros(NP + 8, torch.float64, cfg_o)
    th_ref, s_ref = O.sgd_loop(th.clone(), st, lambda a, z: coupled_forward(a, z, NP), ob, perms, cfg_o.kl_coeff, cfg_o)
    d = torch.from_numpy(g.learner.theta[0].cpu().numpy()).double()
    assert float((d - th_ref).abs().max()) < 1e-3 * float((th_ref - th).abs().max()) + 1e-7
    for k in ("policy_loss", "vf_loss", "kl", "entropy"):
        assert abs(stats[k] - s_ref[k]) < 1e-4 * max(1.0, abs(s_ref[k])), (k, stats[k], s_ref[k])

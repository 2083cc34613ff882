"""GPU: leg-coupled inference in one launch — ddrl_fcnet_forward_coupled (FP32 kernel) and ddrl_fcnet_forward_tc_coupled
(ping-pong tcgen05 kernel), the sampler call and the rollout forward of SharedDecentralLegID (model "cup" = FCNet +
LegCoupling, models/coupling_net_glorot_uniform_init.py:11-30,135).

  * bit for bit equal to the three-launch composition forward -> ddrl_leg_coupling -> ddrl_dg_sample of the same kind;
  * within 1e-5 of the float64 oracle;
  * a node-id column shifted by one leg changes the outputs (negative control); out-of-range ids set DDRL_STATUS_BAD_NODE;
  * FCNetLearner(leg_coupling=True) stores exactly the composition's logits / actions / logp in its rollout buffers, and
    compute_actions / PPOPolicyGroup.compute_actions return exactly the composition."""
import numpy as np
import pytest
import torch

from tests.util import scaled_err

pytestmark = pytest.mark.gpu

TABLE = np.array([[0.7, -1.3], [-0.4, 0.9], [1.6, -0.2], [-1.1, 0.5]], np.float32)   # non-initial: a wrong multiply shows
TOL = 1e-5
FILTERS = {"none": (False, 0.0), "norm": (True, 0.0), "norm-clip10": (True, 10.0)}


def _O():
    import oracle.ddrl_oracle as O
    return O


def _inputs(R, D, seed):
    """theta [1, NP], raw obs [1, R, D] (wide enough for clip 10 to bite), norm [1, 2, D], node ids [1, R] in random order
    covering all four legs, eps [1, R, 2]."""
    O = _O()
    rng = np.random.default_rng(seed)
    theta = O.fcnet_init(D, 4, torch.Generator().manual_seed(seed)).float()
    obs = (rng.standard_normal((1, R, D)) * 3.0 + 0.5).astype(np.float32)
    mean = 0.3 * rng.standard_normal(D)
    inv = 1.0 / (0.2 + rng.random(D))
    norm = np.stack([mean, inv])[None]
    node = (np.arange(R) % 4).astype(np.int32)
    rng.shuffle(node)
    eps = rng.standard_normal((1, R, 2)).astype(np.float32)
    dev = lambda a: torch.as_tensor(np.ascontiguousarray(a)).cuda()
    return {"theta": theta.cuda()[None].contiguous(), "obs": dev(obs), "norm": dev(norm), "node": dev(node[None]),
            "eps": dev(eps), "table": dev(TABLE)}


def _nan(*shape):
    return torch.full(shape, float("nan"), device="cuda")


def _outs(R, D, eps):
    o = {"logits": _nan(1, R, 4), "value": _nan(1, R), "obs_out": _nan(1, R, D)}
    if eps:
        o.update(action=_nan(1, R, 2), logp=_nan(1, R))
    return o


def _composition(kind, x, node, norm, clip, eps, weights):
    """forward (FP32 or tensor-core, no sampling) -> ddrl_leg_coupling -> ddrl_dg_sample: three launches."""
    from ddrl_b200 import kernels as K
    obs = x["obs"]
    R, D = obs.shape[1], obs.shape[2]
    o = _outs(R, D, False)
    if kind == "tc":
        K.fcnet_forward_tc(weights, obs, 2, norm=norm, clip=clip, out=o)
    else:
        K.fcnet_forward(weights, obs, 2, norm=norm, clip=clip, out=o, want_obs_out=True)
    K.leg_coupling_(o["logits"].view(R, 4), node.view(R), x["table"])
    if eps is not None:
        o["action"], o["logp"] = K.dg_sample(o["logits"].view(R, 4), eps.view(R, 2))
        o["action"], o["logp"] = o["action"].view(1, R, 2), o["logp"].view(1, R)
    return o


def _fused(kind, x, node, norm, clip, eps, weights, status=None):
    from ddrl_b200 import kernels as K
    R, D = x["obs"].shape[1], x["obs"].shape[2]
    out = _outs(R, D, eps is not None)
    f = K.fcnet_forward_tc_coupled if kind == "tc" else K.fcnet_forward_coupled
    return f(weights, x["obs"], node, x["table"], 2, norm=norm, clip=clip, eps=eps, status=status, out=out)


def _weights(kind, x):
    from ddrl_b200 import kernels as K
    return K.fcnet_tc_pack(x["theta"], x["obs"].shape[2], 2) if kind == "tc" else x["theta"]


def _assert_equal(got, want, keys):
    for k in keys:
        assert torch.isfinite(got[k]).all(), k
        assert torch.equal(got[k], want[k]), k


@pytest.mark.parametrize("filt", list(FILTERS))
@pytest.mark.parametrize("D", [19, 20])
@pytest.mark.parametrize("R", [1, 7, 129, 4096, 20011, 524288])
@pytest.mark.parametrize("kind", ["fp32", "tc"])
def test_fused_launch_is_the_three_launch_composition_bit_for_bit(kind, R, D, filt):
    use_norm, clip = FILTERS[filt]
    x = _inputs(R, D, seed=R + D)
    norm = x["norm"] if use_norm else None
    w = _weights(kind, x)
    for eps in (x["eps"], None):
        want = _composition(kind, x, x["node"], norm, clip, eps, w)
        status = torch.zeros(1, dtype=torch.int32, device="cuda")
        got = _fused(kind, x, x["node"], norm, clip, eps, w, status=status)
        torch.cuda.synchronize()
        keys = ("logits", "value", "obs_out") + (("action", "logp") if eps is not None else ())
        _assert_equal(got, want, keys)
        assert int(status.item()) & 128 == 0
        if eps is None:
            assert "action" not in got or got["action"] is None


@pytest.mark.parametrize("D", [19, 20])
@pytest.mark.parametrize("R", [7, 4096])
@pytest.mark.parametrize("kind", ["fp32", "tc"])
def test_fused_launch_matches_the_float64_oracle(kind, R, D):
    O = _O()
    x = _inputs(R, D, seed=3 * R + D)
    got = _fused(kind, x, x["node"], x["norm"], 10.0, x["eps"], _weights(kind, x))
    torch.cuda.synchronize()
    h = lambda t: t[0].cpu().double()
    raw, nm = h(x["obs"]), x["norm"][0].cpu()
    xin = ((raw - nm[0]) * nm[1]).clamp(-10.0, 10.0)
    assert scaled_err(h(got["obs_out"]), xin) < 1e-6
    lg, v = O.fcnet_forward(x["theta"][0].cpu().double(), h(got["obs_out"]), 4)
    lg = O.leg_coupling(lg, x["node"][0].cpu().long(), torch.from_numpy(TABLE).double())
    act = O.dg_sample(lg, h(x["eps"]))
    logp = O.dg_logp(lg, act)
    for name, ref in (("logits", lg), ("value", v), ("action", act), ("logp", logp)):
        assert scaled_err(h(got[name]).numpy(), ref.numpy()) < TOL, (kind, name)


@pytest.mark.parametrize("kind", ["fp32", "tc"])
def test_shifted_node_ids_change_the_outputs(kind):
    x = _inputs(4096, 19, seed=11)
    w = _weights(kind, x)
    want = _composition(kind, x, x["node"], x["norm"], 0.0, x["eps"], w)
    got = _fused(kind, x, ((x["node"] + 1) % 4).contiguous(), x["norm"], 0.0, x["eps"], w)
    torch.cuda.synchronize()
    for k in ("logits", "action", "logp"):
        assert not torch.equal(got[k], want[k]), k
    assert torch.equal(got["value"], want["value"])


@pytest.mark.parametrize("kind", ["fp32", "tc"])
def test_out_of_range_node_ids_set_the_status_bit(kind):
    x = _inputs(1000, 19, seed=5)
    w = _weights(kind, x)
    bad = x["node"].clone()
    bad[0, 3], bad[0, 700] = 4, -1
    status = torch.zeros(1, dtype=torch.int32, device="cuda")
    got = _fused(kind, x, bad, x["norm"], 0.0, x["eps"], w, status=status)
    want = _composition(kind, x, (bad & 3).contiguous(), x["norm"], 0.0, x["eps"], w)     # bad rows: coupled as id & 3
    torch.cuda.synchronize()
    assert int(status.item()) & 128
    _assert_equal(got, want, ("logits", "value", "obs_out", "action", "logp"))
    ok = torch.ones(1000, dtype=torch.bool, device="cuda")
    ok[3] = ok[700] = False
    ref = _composition(kind, x, x["node"], x["norm"], 0.0, x["eps"], w)      # every other row as with valid ids
    for k in ("logits", "action", "logp"):
        assert torch.equal(got[k][0][ok], ref[k][0][ok]), k


def test_entries_reject_bad_arguments():
    from ddrl_b200 import _lib
    from ddrl_b200 import kernels as K
    lib = _lib.load()
    x = _inputs(64, 19, seed=1)
    img = K.fcnet_tc_pack(x["theta"], 19, 2)
    st = torch.zeros(1, dtype=torch.int32, device="cuda")
    lg, v = _nan(2, 64, 16), _nan(2, 64)
    obs27 = torch.zeros(1, 64, 27, device="cuda")
    p = lambda t: None if t is None else t.data_ptr()

    def fp(status=st, P=1, A=2, R=64, obs=x["obs"], D=19):
        return lib.ddrl_fcnet_forward_coupled(p(x["theta"]), None, p(x["node"]), p(x["table"]), p(obs), None, 0.0, P, R, D, A,
                                              None, p(lg), p(v), None, None, None, p(status), None)

    def tc(status=st, P=1, A=2, R=64, obs=x["obs"], D=19):
        return lib.ddrl_fcnet_forward_tc_coupled(p(img), p(x["node"]), p(x["table"]), p(obs), None, 0.0, P, R, D, A, None,
                                                 p(lg), p(v), None, None, None, p(status), None)

    for f in (fp, tc):
        assert f(status=None) == -1 and b"status" in lib.ddrl_last_error()
        assert f(A=4) == -1 and b"A = 2" in lib.ddrl_last_error()
        assert f(P=2) == -1 and b"P = 1" in lib.ddrl_last_error()
        assert f(R=-1) == -1
        assert f(R=0) == 0
    assert tc(obs=obs27, D=27) == -2 and b"D = 19 or 20" in lib.ddrl_last_error()
    torch.cuda.synchronize()
    assert int(st.item()) == 0 and torch.isnan(lg).all()      # nothing was launched


# ---- the learner and the policy group ---------------------------------------------------------------------------------

def _theta0():
    O = _O()
    th = O.fcnet_init(19, 4, torch.Generator().manual_seed(7))
    return torch.cat([th, torch.from_numpy(TABLE.reshape(-1))])


@pytest.mark.parametrize("mode", ["tc", "fp32"])
def test_learner_rollout_buffers_are_the_composition(mode):
    """After one learn_on_rollout the unshuffled logits / act / logp buffers equal forward -> leg_coupling -> dg_sample,
    recomputed from the learner's own filtered obs buffer and the rollout's noise with the pre-update weights."""
    from ddrl_b200 import kernels as K
    from ddrl_b200.config import PPOConfig
    from ddrl_b200.learner import FCNetLearner
    th0 = _theta0()
    L = FCNetLearner(1, 19, 2, PPOConfig(num_sgd_iter=2, sgd_minibatch_size=128), "cuda", theta=th0[None], mode=mode,
                     leg_coupling=True)
    rng = np.random.default_rng(4)
    T, N = 16, 8
    C, R = 4 * N, 16 * 4 * N
    to = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    raw = (rng.standard_normal((1, T, C, 19)) * 2.0 + 0.5).astype(np.float32)
    boot = (rng.standard_normal((1, C, 19)) * 2.0 + 0.5).astype(np.float32)
    rew = (0.3 + 0.5 * rng.standard_normal((1, T, C))).astype(np.float32)
    dones = (rng.random((T, N)) < 0.05).astype(np.uint8)
    eps = rng.standard_normal((1, T, C, 2)).astype(np.float32)
    perms = np.stack([rng.permutation(R // 128) for _ in range(2)])[None].astype(np.int32)
    L.learn_on_rollout(to(raw), to(boot), to(rew), to(dones), to(eps), to(perms), shuffle=to(rng.permutation(R).astype(np.int32)[None]),
                       cols_per_env=4)
    torch.cuda.synchronize()
    b = L._bufs
    NP = th0.numel() - 8
    x = {"obs": b["obs"].clone(), "table": th0[NP:].cuda().reshape(4, 2).contiguous()}
    theta_fc = th0[:NP].cuda()[None].contiguous()
    w = K.fcnet_tc_pack(theta_fc, 19, 2) if mode == "tc" else theta_fc
    want = _composition(mode, x, b["node"], None, 0.0, to(eps).reshape(1, R, 2), w)
    torch.cuda.synchronize()
    assert not torch.equal(L.theta[0].cpu(), th0)      # the update ran after the forward
    for k, bk in (("logits", "logits"), ("action", "act"), ("logp", "logp")):
        assert torch.equal(b[bk], want[k]), k


def test_compute_actions_is_the_composition():
    from ddrl_b200 import kernels as K
    from ddrl_b200._lib import DDRLError
    from ddrl_b200.config import PPOConfig
    from ddrl_b200.learner import FCNetLearner
    th0 = _theta0()
    L = FCNetLearner(1, 19, 2, PPOConfig(), "cuda", theta=th0[None], leg_coupling=True)
    rng = np.random.default_rng(8)
    NP = th0.numel() - 8
    x = {"table": L.theta[0, NP:]}
    for B, update in ((16, True), (300, False), (16384, False)):
        raw = torch.from_numpy((rng.standard_normal((1, B, 19)) * 2.0).astype(np.float32)).cuda()
        node = torch.from_numpy(rng.integers(0, 4, (1, B)).astype(np.int32)).cuda()
        eps = torch.from_numpy(rng.standard_normal((1, B, 2)).astype(np.float32)).cuda()
        for e in (eps, None):
            got = L.compute_actions(raw, e, update_filter=update and e is not None, node_idx=node)
            x["obs"] = raw
            want = _composition("fp32", x, node, L.norm, L.cfg.filter_clip, e, L.theta_fc.contiguous())
            torch.cuda.synchronize()
            assert set(got) == ({"logits", "value", "action", "logp"} if e is not None else {"logits", "value"})
            _assert_equal(got, want, got.keys())
    node[0, 5] = 4
    with pytest.raises(DDRLError, match="node ids must be 0..3"):
        L.compute_actions(raw, eps, node_idx=node)
    node[0, 5] = -1
    with pytest.raises(DDRLError, match="node ids must be 0..3"):
        L.compute_actions(raw, None, node_idx=node)


@pytest.mark.parametrize("explore", [True, False])
def test_policy_group_compute_actions_is_the_composition(explore):
    from ddrl_b200.rllib_policy import BatchError, PPOPolicyGroup
    g = PPOPolicyGroup("QuantrupedMultiEnv_SharedDecentralLegID", {"sgd_minibatch_size": 128, "num_sgd_iter": 2}, seed=0)
    pid = g.policy_names[0]
    w = g.get_weights()
    w[pid][f"{pid}/leg_coupling"] = TABLE.copy()
    g.set_weights(w)
    rng = np.random.default_rng(3)
    for B in (16, 300):
        obs = rng.standard_normal((B, 19)).astype(np.float32)
        node = rng.integers(0, 4, B)
        state = np.random.RandomState(0)
        state.set_state(g.rng.get_state())
        out = g.compute_actions({pid: (node, obs)}, explore=explore)[pid]
        noise = state.standard_normal((1, B, 2)).astype(np.float32) if explore else np.zeros((1, B, 2), np.float32)
        L = g.learner
        NP = L.theta.shape[1] - 8
        x = {"obs": torch.from_numpy(obs[None]).cuda(), "table": L.theta[0, NP:]}
        use_norm = L.norm if int(L.filt_n.max().item()) > 0 else None
        want = _composition("fp32", x, torch.from_numpy(node[None].astype(np.int32)).cuda(), use_norm, L.cfg.filter_clip,
                            torch.from_numpy(noise).cuda(), L.theta_fc.contiguous())
        h = lambda k: want[k][0].cpu().numpy()
        assert np.array_equal(out[0], h("action"))
        assert np.array_equal(out[2]["action_dist_inputs"], h("logits"))
        assert np.array_equal(out[2]["action_logp"], h("logp"))
        assert np.array_equal(out[2]["vf_preds"], h("value"))
    with pytest.raises(BatchError):
        g.compute_actions({pid: (np.full(16, 4), rng.standard_normal((16, 19)).astype(np.float32))}, explore=explore)

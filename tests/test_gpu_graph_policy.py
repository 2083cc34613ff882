"""GPU: the shared GraphNet policy through the RLlib-facing surface — `ddrl_graphnet_act` (GraphNet forward + DiagGaussian
sample in one launch) against the two-launch path and the oracle, `GraphNetLearner.compute_actions`, and
`rllib_policy.GraphNetPolicyGroup` (compute_actions / postprocess_fragments / learn_on_batch / weights) against the oracle's
restatement of the same RLlib steps."""
import numpy as np
import pytest
import torch

from tests.test_gpu_graphnet import _O, _dev, _inputs, _theta
from tests.util import scaled_err

pytestmark = pytest.mark.gpu
SCOPE = "QuantrupedMultiEnv_DecentralShared_Graph"


def _close(a, b):
    """Within 1e-5 of the reference's scale, or 1e-6 absolute: one near-zero value (B = 1) is its own scale, and the
    GraphNet's MUFU tanh has an absolute error of up to 2.4e-7."""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return scaled_err(a, b) < 1e-5 or np.abs(a - b).max() < 1e-6


def _graph_inputs(B, seed, adj_kind):
    if adj_kind == "zero":
        idx, state, adj = _inputs(B, seed, "ring")
        return idx, state, np.zeros_like(adj)
    return _inputs(B, seed, adj_kind)


@pytest.mark.parametrize("adj_kind", ["ring", "random", "zero"])
@pytest.mark.parametrize("A", [2, 4, 8])
@pytest.mark.parametrize("B", [1, 7, 257, 20011])
def test_graphnet_act_is_forward_plus_dg_sample_bit_for_bit(B, A, adj_kind):
    from ddrl_b200 import kernels as K
    O = _O()
    idx, state, adj = _graph_inputs(B, 3 * B + A, adj_kind)
    th = _theta(A, 1, big=True)
    rng = np.random.default_rng(B + A)
    eps = rng.standard_normal((B, A)).astype(np.float32)
    d_th, d_idx, d_st, d_adj, d_eps = _dev(th.numpy(), torch.float32), _dev(idx), _dev(state), _dev(adj), _dev(eps)
    nan = lambda *shape: torch.full(shape, float("nan"), device="cuda")
    K.graphnet_set_variant(1)
    try:
        lg, v = K.graphnet_forward(d_th, d_idx, d_st, d_adj, A, out=(nan(B, 2 * A), nan(B)))
        act, logp = K.dg_sample(lg, d_eps)
        fused = K.graphnet_act(d_th, d_idx, d_st, d_adj, d_eps, A, out=(nan(B, 2 * A), nan(B), nan(B, A), nan(B)))
        mean = K.graphnet_act(d_th, d_idx, d_st, d_adj, torch.zeros_like(d_eps), A)
        torch.cuda.synchronize()
    finally:
        K.graphnet_set_variant(-1)
    for want, got in zip((lg, v, act, logp), fused):
        assert torch.isfinite(got).all()
        assert torch.equal(want, got)
    assert torch.equal(mean[0], lg) and torch.equal(mean[2], lg[:, :A])          # zero noise: the action is the mean
    # float64 oracle (the device sees float32 weights)
    lg_ref, v_ref = O.graphnet_forward(th.float().double(), torch.from_numpy(idx), torch.from_numpy(state).double(),
                                       torch.from_numpy(adj).double(), 2 * A)
    act_ref = O.dg_sample(lg_ref, torch.from_numpy(eps).double())
    assert _close(fused[0].cpu().numpy(), lg_ref.numpy())
    assert _close(fused[1].cpu().numpy(), v_ref.numpy())
    assert _close(fused[2].cpu().numpy(), act_ref.numpy())
    assert _close(fused[3].cpu().numpy(), O.dg_logp(lg_ref, act_ref).numpy())


def test_graphnet_learner_compute_actions():
    from ddrl_b200 import kernels as K
    from ddrl_b200._lib import DDRLError
    from ddrl_b200.config import PPOConfig
    from ddrl_b200.learner import GraphNetLearner
    A, B = 2, 300
    idx, state, adj = _inputs(B, 5, "random")
    eps = np.random.default_rng(6).standard_normal((B, A)).astype(np.float32)
    th = _theta(A, 2, big=True).float()
    L = GraphNetLearner(A, PPOConfig(), "cuda", theta=th.reshape(1, -1))
    d_idx, d_st, d_adj, d_eps = _dev(idx), _dev(state), _dev(adj), _dev(eps)
    K.graphnet_set_variant(1)
    try:
        lg, v = K.graphnet_forward(_dev(th.numpy()), d_idx, d_st, d_adj, A)
        act, logp = K.dg_sample(lg, d_eps)
        res = L.compute_actions(d_idx, d_st, d_adj, d_eps)
        plain = L.compute_actions(d_idx, d_st, d_adj)
        torch.cuda.synchronize()
    finally:
        K.graphnet_set_variant(-1)
    assert set(res) == {"logits", "value", "action", "logp"} and set(plain) == {"logits", "value"}
    for k, want in (("logits", lg), ("value", v), ("action", act), ("logp", logp)):
        assert torch.equal(res[k], want), k
    assert torch.equal(plain["logits"], lg) and torch.equal(plain["value"], v)
    for bad in (4, -1):
        b_idx = d_idx.clone()
        b_idx[B // 2] = bad
        with pytest.raises(DDRLError, match="0..3"):
            L.compute_actions(b_idx, d_st, d_adj, d_eps)


def _weights(pid, th, A):
    from ddrl_b200.modelv2 import graphnet_shapes
    out, o = {}, 0
    for name, shp in graphnet_shapes(2 * A):
        n = int(np.prod(shp))
        out[f"{pid}/{name}"] = th[o:o + n].reshape(shp)
        o += n
    return out


@pytest.mark.parametrize("step", ["tc", "three-kernel"])
def test_graph_policy_group_serves_the_rllib_calls(step):
    import oracle.ddrl_oracle as O
    from ddrl_b200 import rllib_policy as RP
    A, T, N, E, MB, SEED = 2, 10, 13, 2, 128, 3
    C = 4 * N
    R = T * C                                              # 520 rows: 4 whole minibatches of 128 + a ragged tail of 8
    cfg = {"num_sgd_iter": E, "sgd_minibatch_size": MB, "seed": SEED}
    g = RP.GraphNetPolicyGroup(SCOPE, cfg, step=step)
    pid = g.policy_names[0]
    assert g.policy_names == ["leg_policy"] and g.A == A
    th0 = _theta(A, 5, big=True).float().numpy()
    w0 = _weights(pid, th0, A)
    g.set_weights({pid: w0})
    w = g.get_weights()
    assert list(w) == [pid] and list(w[pid]) == list(w0)
    assert w[pid][f"{pid}/actor/state_enc/kernel"].shape == (4, 19 * 64)
    assert w[pid][f"{pid}/critic/linear_out/bias"].shape == (1,)
    assert all(np.array_equal(w[pid][k], w0[k]) for k in w0)
    assert np.array_equal(g.learner.theta.cpu().numpy().reshape(-1), th0)

    rng = np.random.default_rng(4)
    idx = np.tile(np.arange(4, dtype=np.int32), R // 4)             # env-major leg columns FL, HL, HR, FR
    _, state, adj = _inputs(R, 41, "ring")
    adj[: R // 4] = (rng.random((R // 4, 4, 4)) < 0.4)               # some rows with other 0/1 graphs
    state = state.astype(np.float64)                                # the env's Box is float64
    bidx = np.tile(np.arange(4, dtype=np.int32), N)
    _, bstate, badj = _inputs(C, 42, "ring")
    rewards = (0.3 + 0.5 * rng.standard_normal((1, T, C))).astype(np.float32)
    dones = np.repeat(rng.random((T, N)) < 0.1, 4, axis=1).astype(np.uint8)

    # ---- compute_actions -------------------------------------------------------------------------------------------
    out = g.compute_actions({pid: (idx, state, adj)})
    last = g.compute_actions({pid: (bidx[:, None], bstate, badj)}, explore=False)
    replay = np.random.RandomState(SEED)
    noise = replay.standard_normal((1, R, A)).astype(np.float32)
    act, st_, info = out[pid]
    assert st_ == [] and act.shape == (R, A) and set(info) == {RP.ACTION_DIST_INPUTS, RP.ACTION_LOGP, RP.VF_PREDS}
    t32 = lambda a: torch.from_numpy(np.asarray(a, dtype=np.float32)).double()
    logits, value = O.graphnet_forward(torch.from_numpy(th0).double(), torch.from_numpy(idx), t32(state), t32(adj), 2 * A)
    want_act = O.dg_sample(logits, torch.from_numpy(noise[0]).double())
    assert scaled_err(info[RP.ACTION_DIST_INPUTS], logits.numpy()) < 1e-5
    assert scaled_err(info[RP.VF_PREDS], value.numpy()) < 1e-5
    assert scaled_err(act, want_act.numpy()) < 1e-5
    assert scaled_err(info[RP.ACTION_LOGP], O.dg_logp(logits, want_act).numpy()) < 1e-5
    assert np.array_equal(last[pid][0], last[pid][2][RP.ACTION_DIST_INPUTS][:, :A])     # explore=False: the mean

    # ---- postprocess_fragments ---------------------------------------------------------------------------------------------
    vf = info[RP.VF_PREDS].reshape(1, T, C)
    last_v = last[pid][2][RP.VF_PREDS].reshape(1, C)
    adv, vt = g.postprocess_fragments(rewards, vf, dones, last_v)
    a_ref, v_ref = O.gae_recurrence(rewards[0], vf[0], dones, last_v[0], 0.99, 0.95)
    assert scaled_err(adv[0], a_ref) < 1e-5 and scaled_err(vt[0], v_ref) < 1e-5

    # ---- learn_on_batch ----------------------------------------------------------------------------------------------
    batch = {RP.NODE_IDX: idx, RP.OBS: state, RP.ADJ: adj, RP.ACTIONS: act, RP.ACTION_DIST_INPUTS: info[RP.ACTION_DIST_INPUTS],
             RP.ACTION_LOGP: info[RP.ACTION_LOGP], RP.VF_PREDS: info[RP.VF_PREDS], RP.ADVANTAGES: adv[0].reshape(-1),
             RP.VALUE_TARGETS: vt[0].reshape(-1)}
    rng_state = g.rng.get_state()
    res = g.learn_on_batch({pid: batch})
    assert g.num_steps_trained == 512 and set(res) == {pid}
    shuffle, perms = RP.draw_minibatch_order(replay, 1, R, E, 4)      # the draws the group made after the action noise
    cfg_o = O.PPOConfig(num_sgd_iter=E, sgd_minibatch_size=MB)
    fwd = lambda th, obs: O.graphnet_forward(th, obs[0], obs[1], obs[2], 2 * A)
    rows = shuffle[0][:512].astype(np.int64)
    adv_std = O.standardized(np.asarray(batch[RP.ADVANTAGES], dtype=np.float32))           # over all 520 rows

    def oracle(dt, reorder=None):
        r = rows
        if reorder is not None:     # the same minibatches with their rows in another order: the same update in float64
            rr = np.random.default_rng(reorder)
            r = np.concatenate([rr.permutation(rows[k * MB:(k + 1) * MB]) for k in range(4)])
        t = lambda a: torch.from_numpy(np.asarray(a, dtype=np.float32)[r]).to(dt)
        ti, ts, ta = torch.from_numpy(idx[r]), t(state), t(adj)

        class _Obs:  # row-sliceable tuple observation
            def __getitem__(self, sl):
                return (ti[sl], ts[sl], ta[sl])
        ob = {"obs": _Obs(), "actions": t(batch[RP.ACTIONS]), "old_logits": t(batch[RP.ACTION_DIST_INPUTS]),
              "old_logp": t(batch[RP.ACTION_LOGP]), "vf_preds": t(batch[RP.VF_PREDS]), "advantages": t(adv_std),
              "value_targets": t(batch[RP.VALUE_TARGETS])}
        return O.sgd_loop(torch.from_numpy(th0).to(dt), O.AdamState.zeros(th0.size, dt, cfg_o), fwd, ob, perms[0],
                          cfg_o.kl_coeff, cfg_o)
    th64, ref_stats = oracle(torch.float64)
    got = g.learner.theta.cpu().numpy().reshape(-1).astype(np.float64)
    upd = th64.numpy() - th0
    err_dev = scaled_err(got - th0, upd)
    # the float32 twin's distance from float64 depends on the summation order (here 4e-5 .. 2e-4 of the update over row
    # orders within the minibatches), so the device is held to 10x the largest of a few orders
    err_twin = max(scaled_err(oracle(torch.float32, k)[0].numpy().astype(np.float64) - th0, upd) for k in (None, 1, 2, 3))
    assert err_dev < 10.0 * err_twin + 1e-5, (err_dev, err_twin)     # no further from float64 than 10x the float32 twin
    assert scaled_err(got, th64.numpy()) < 2e-3
    ls = res[pid]["learner_stats"]
    for k in ("total_loss", "policy_loss", "vf_loss", "kl", "entropy", "vf_explained_var"):
        assert abs(ls[k] - ref_stats[k]) < 1e-4 * max(1.0, abs(ref_stats[k])), (k, ls[k], ref_stats[k])
    assert {"cur_kl_coeff", "cur_lr"} <= set(ls)
    moved = g.get_weights()[pid]
    assert not np.array_equal(moved[f"{pid}/actor/linear_out/kernel"], w0[f"{pid}/actor/linear_out/kernel"])

    # ---- same seed, same batch: bit-identical (the GraphNet steps reduce in fixed order) ---------------------------------
    g2 = RP.GraphNetPolicyGroup(SCOPE, cfg, step=step)
    g2.set_weights({pid: w0})
    g2.rng.set_state(rng_state)
    res2 = g2.learn_on_batch({pid: batch})
    assert torch.equal(g.learner.theta, g2.learner.theta) and torch.equal(g.learner.m, g2.learner.m)
    assert res2 == res


def test_graph_policy_group_fails_loudly():
    from ddrl_b200 import _lib
    from ddrl_b200 import checkpoint as CK
    from ddrl_b200 import rllib_policy as RP
    g = RP.GraphNetPolicyGroup(SCOPE, {"sgd_minibatch_size": 8, "num_sgd_iter": 1})
    pid = g.policy_names[0]
    B = 16
    idx, state, adj = _inputs(B, 9, "ring")
    ok = (idx, state, adj)
    bad_cases = {
        "node id": (np.full(B, 4), state, adj),
        "adj = 2": (idx, state, adj * 2),
        "NaN state": (idx, np.where(np.arange(23) == 5, np.nan, state), adj),
        "state shape": (idx, state[:, :, :19], adj),
    }
    for what, tup in bad_cases.items():
        with pytest.raises(RP.BatchError):
            g.compute_actions({pid: tup})
    out = g.compute_actions({pid: ok})[pid]
    batch = {RP.NODE_IDX: idx, RP.OBS: state, RP.ADJ: adj, RP.ACTIONS: out[0], RP.ACTION_DIST_INPUTS: out[2][RP.ACTION_DIST_INPUTS],
             RP.ACTION_LOGP: out[2][RP.ACTION_LOGP], RP.VF_PREDS: out[2][RP.VF_PREDS], RP.ADVANTAGES: np.ones(B, np.float32),
             RP.VALUE_TARGETS: np.zeros(B, np.float32)}
    for what, change in (("node id", {RP.NODE_IDX: np.full(B, -1)}), ("adj = 2", {RP.ADJ: adj * 2}),
                         ("NaN state", {RP.OBS: np.where(np.arange(23) == 5, np.nan, state)}),
                         ("state shape", {RP.OBS: state[:, :3]}), ("ragged", {RP.VF_PREDS: out[2][RP.VF_PREDS][:-1]})):
        with pytest.raises(RP.BatchError):
            g.learn_on_batch({pid: dict(batch, **change)})
    with pytest.raises(RP.BatchError, match="adj"):
        g.learn_on_batch({pid: {k: v for k, v in batch.items() if k != RP.ADJ}})
    with pytest.raises(ValueError):
        g.set_weights({pid: {k: v for i, (k, v) in enumerate(g.get_weights()[pid].items()) if i}})
    with pytest.raises(NotImplementedError, match="target"):
        RP.GraphNetPolicyGroup(SCOPE, use_target_velocity=True)
    with pytest.raises(NotImplementedError, match="19"):
        RP.GraphNetPolicyGroup("QuantrupedMultiEnv_Decentral_Graph")
    with pytest.raises(ValueError, match="PPOPolicyGroup"):
        RP.GraphNetPolicyGroup("QuantrupedMultiEnv_FullyDecentral")
    with pytest.raises(ValueError, match="get_weights"):
        CK.from_learner(g.learner, [pid])
    with pytest.raises(ValueError, match="get_weights"):
        CK.apply_to_learner(None, g.learner)
    lib = _lib.load()
    p = torch.zeros(4096, device="cuda")
    ptr = p.data_ptr()
    assert lib.ddrl_graphnet_act(ptr, None, ptr, ptr, ptr, 1, 2, ptr, ptr, ptr, ptr, None) == -1      # DDRL_E_BADARG
    assert b"graphnet_act" in lib.ddrl_last_error()
    for A in (0, 9):
        assert lib.ddrl_graphnet_act(ptr, ptr, ptr, ptr, ptr, 1, A, ptr, ptr, ptr, ptr, None) == -2  # DDRL_E_UNSUPPORTED_SHAPE
    assert lib.ddrl_graphnet_act(ptr, ptr, ptr, ptr, ptr, -1, 2, ptr, ptr, ptr, ptr, None) == -1
    assert lib.ddrl_graphnet_act(ptr, ptr, ptr, ptr, ptr, 0, 2, ptr, ptr, ptr, ptr, None) == 0        # B == 0: no-op

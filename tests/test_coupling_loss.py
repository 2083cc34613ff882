"""CPU: the coupled PPO loss of SharedDecentralLegID (FCNet + LegCoupling) that the leg-coupled SGD steps are checked
against — float64 finite differences of the table gradient, and the table == 1 identity with the plain FCNet loss."""
import numpy as np
import torch

import oracle.ddrl_oracle as O

D, A = 19, 2


def _setup(R=96, seed=0):
    g = torch.Generator().manual_seed(seed)
    rng = np.random.default_rng(seed)
    theta = O.fcnet_init(D, 2 * A, g).double()
    x = torch.from_numpy(rng.standard_normal((R, D)))
    node = torch.from_numpy(rng.integers(0, 4, R).astype(np.int32))
    lg, _ = O.fcnet_forward(theta, x, 2 * A)
    old = lg + 0.05 * torch.from_numpy(rng.standard_normal(lg.shape))
    act = old[:, :A] + torch.exp(old[:, A:]) * torch.from_numpy(rng.standard_normal((R, A)))
    batch = {"x": x, "node": node, "act": act, "old": old, "old_logp": O.dg_logp(old, act),
             "vf": torch.from_numpy(rng.standard_normal(R)), "adv": torch.from_numpy(rng.standard_normal(R)),
             "vt": torch.from_numpy(rng.standard_normal(R))}
    return theta, batch


def _loss(theta, table, b, cfg, coupled=True):
    lg, v = O.fcnet_forward(theta, b["x"], 2 * A)
    if coupled:
        lg = O.leg_coupling(lg, b["node"], table)
    loss, _ = O.ppo_loss_from_outputs(lg, v, b["act"], b["old"], b["old_logp"], b["vf"], b["adv"], b["vt"], 0.3, cfg)
    return loss


def test_table_gradient_matches_finite_differences():
    cfg = O.PPOConfig(entropy_coeff=0.01)
    theta, b = _setup()
    table = torch.tensor([[0.7, -1.3], [-0.4, 0.9], [1.6, -0.2], [-1.1, 0.5]], dtype=torch.float64, requires_grad=True)
    (g,) = torch.autograd.grad(_loss(theta, table, b, cfg), table)
    h = 1e-6
    fd = torch.zeros(4, 2, dtype=torch.float64)
    with torch.no_grad():
        for n in range(4):
            for i in range(2):
                tp, tm = table.detach().clone(), table.detach().clone()
                tp[n, i] += h
                tm[n, i] -= h
                fd[n, i] = (_loss(theta, tp, b, cfg) - _loss(theta, tm, b, cfg)) / (2 * h)
    assert torch.allclose(g, fd, rtol=1e-6, atol=1e-9), (g, fd)
    # the closed form the kernels implement: d c[n][i] = sum_{r: node = n} dlogits[r][i] * pre[r][i]
    lg_pre, _ = O.fcnet_forward(theta, b["x"], 2 * A)
    lg_pre = lg_pre.detach()
    lg = O.leg_coupling(lg_pre, b["node"], table.detach()).requires_grad_(True)
    _, v = O.fcnet_forward(theta, b["x"], 2 * A)
    loss, _ = O.ppo_loss_from_outputs(lg, v.detach(), b["act"], b["old"], b["old_logp"], b["vf"], b["adv"], b["vt"], 0.3, cfg)
    (dl,) = torch.autograd.grad(loss, lg)
    closed = torch.zeros(4, 2, dtype=torch.float64)
    for n in range(4):
        sel = b["node"].long() == n
        closed[n] = (dl[sel, :2] * lg_pre[sel, :2]).sum(0)
    assert torch.allclose(g, closed, rtol=1e-12, atol=1e-15)


def test_table_of_ones_equals_the_uncoupled_loss():
    cfg = O.PPOConfig(entropy_coeff=0.01)
    theta, b = _setup(seed=3)
    th = theta.clone().requires_grad_(True)
    ones = torch.ones(4, 2, dtype=torch.float64)
    lc = _loss(th, ones, b, cfg)
    (gc,) = torch.autograd.grad(lc, th)
    th2 = theta.clone().requires_grad_(True)
    lu = _loss(th2, ones, b, cfg, coupled=False)
    (gu,) = torch.autograd.grad(lu, th2)
    assert float(lc) == float(lu)
    assert torch.equal(gc, gu)


def test_coupled_oracle_step_with_unit_table_equals_the_uncoupled_step():
    """The coupled forward of tests/coupling_oracle.py, run through the oracle's own sgd_minibatch_step with the table == 1,
    gives the FCNet step bit for bit in float64 (grad_clip large, so that the table's own gradient — nonzero even at 1 —
    cannot change the clip scale; the table has its own Adam state)."""
    from tests.coupling_oracle import coupled_forward
    R = 64
    rng = np.random.default_rng(0)
    th = O.fcnet_init(D, 2 * A, torch.Generator().manual_seed(1)).double()
    NP = th.numel()
    x = torch.from_numpy(rng.standard_normal((R, D)))
    xx = torch.cat([(torch.arange(R) % 4).double()[:, None], x], 1)
    cfg = O.PPOConfig(grad_clip=1e9, sgd_minibatch_size=R, entropy_coeff=0.01)
    lg, v = O.fcnet_forward(th, x, 2 * A)
    act = O.dg_sample(lg, torch.from_numpy(rng.standard_normal((R, A))))
    b = {"actions": act, "old_logits": lg + 0.01, "old_logp": O.dg_logp(lg + 0.01, act), "vf_preds": v,
         "advantages": torch.from_numpy(rng.standard_normal(R)), "value_targets": v + 1}
    su, sc = O.AdamState.zeros(NP, torch.float64, cfg), O.AdamState.zeros(NP + 8, torch.float64, cfg)
    tu, stu, gu, _ = O.sgd_minibatch_step(th, su, lambda t, z: O.fcnet_forward(t, z, 2 * A), dict(b, obs=x), slice(0, R), 0.2, cfg)
    tc, stc, gc, _ = O.sgd_minibatch_step(torch.cat([th, torch.ones(8, dtype=torch.float64)]), sc,
                                          lambda t, z: coupled_forward(t, z, NP), dict(b, obs=xx), slice(0, R), 0.2, cfg)
    assert torch.equal(gc[:NP], gu) and torch.equal(tc[:NP], tu)
    assert torch.equal(sc.m[:NP], su.m) and torch.equal(sc.v[:NP], su.v) and stc == stu


def test_policy_group_validates_the_node_idx_column():
    import pytest
    from ddrl_b200.rllib_policy import BatchError, check_node_idx
    assert check_node_idx(np.array([0, 1, 2, 3, 3]), 5, "x").dtype == np.int32
    assert check_node_idx(np.array([[1.0], [2.0]]), 2, "x").tolist() == [1, 2]
    for bad, rows in ((np.array([0, 4]), 2), (np.array([-1, 0]), 2), (np.array([0, 1]), 3), (np.array([0.5, 1.0]), 2),
                      (np.zeros((2, 2), np.int64), 2)):
        with pytest.raises(BatchError):
            check_node_idx(bad, rows, "x")

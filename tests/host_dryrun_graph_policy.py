"""Host-logic dry run of `rllib_policy.GraphNetPolicyGroup` (CPU, own process — it monkeypatches torch; run by
tests/test_graph_policy_host.py).

The fused kernel (`K.graphnet_act`), the GraphNet forward, GAE and StandardizeFields are replaced by the ORACLE's float64
restatement, the learner's SGD phase by the oracle's float32 `sgd_loop`, "cuda" is mapped to "cpu", and the GPU test of
the group's RLlib calls (tests/test_gpu_graph_policy.py) is executed unchanged for both step kinds.  It checks the
orchestration — the RandomState draw order, StandardizeFields over the whole batch before the ragged tail is dropped, the
rows handed to the learner, the weight names — and no kernel.  Test infrastructure only."""
import os
import sys
import types

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import oracle.ddrl_oracle as O  # noqa: E402

_dev = torch.device
torch.device = lambda *a, **k: _dev("cpu")
torch.cuda.is_available = lambda: True
torch.cuda.get_device_properties = lambda d: types.SimpleNamespace(multi_processor_count=148)
torch.cuda.synchronize = lambda *a: None
torch.Tensor.cuda = lambda self, *a, **k: self
torch.Tensor.is_cuda = property(lambda self: True)

import ddrl_b200.kernels as K  # noqa: E402
import ddrl_b200.learner as L  # noqa: E402

D64 = lambda t: t.detach().double()       # noqa: E731
CALLS = []


def graphnet_forward(theta, idx, st, adj, A, out=None):
    CALLS.append("graphnet_forward")
    lg, v = O.graphnet_forward(D64(theta).reshape(-1), idx, D64(st), D64(adj), 2 * A)
    return lg.float(), v.float()


def graphnet_act(theta, idx, st, adj, eps, A, out=None):
    CALLS.append("graphnet_act")
    lg, v = O.graphnet_forward(D64(theta).reshape(-1), idx, D64(st), D64(adj), 2 * A)
    a = O.dg_sample(lg, D64(eps))
    return lg.float(), v.float(), a.float(), O.dg_logp(lg, a).float()


def gae(rewards, values, dones, v_boot, cpe, gamma, lam, adv=None, vtarg=None, moments=None, ws=None):
    P = rewards.shape[0]
    adv, vtarg = torch.empty_like(rewards), torch.empty_like(rewards)
    moments = torch.empty(P, 3, dtype=torch.float64)
    dn = np.repeat(dones.numpy(), cpe, axis=1)
    for p in range(P):
        a, v = O.gae_recurrence(rewards[p].numpy(), values[p].numpy(), dn, v_boot[p].numpy(), gamma, lam)
        adv[p], vtarg[p] = torch.from_numpy(a.astype(np.float32)), torch.from_numpy(v.astype(np.float32))
        a64 = a.astype(np.float32).astype(np.float64)
        moments[p] = torch.tensor([a64.size, a64.sum(), (a64 ** 2).sum()])
    return adv, vtarg, moments


def adv_standardize(adv, moments):
    CALLS.append(("adv_standardize", int(moments[0, 0])))
    P = adv.shape[0]
    flat = adv.view(P, -1)
    mean = moments[:, 1] / moments[:, 0]
    std = (moments[:, 2] / moments[:, 0] - mean ** 2).clamp_min(0).sqrt().clamp_min(1e-4)
    flat.copy_(((flat.double() - mean[:, None]) / std[:, None]).float())
    return adv


def sgd_phase(self, cols, perms, shuffle, R):
    # the group hands over the truncated batch in shuffled order: no shuffle left, whole minibatches only
    MB = self.cfg.sgd_minibatch_size
    assert shuffle is None and R % MB == 0 and tuple(perms.shape) == (self.cfg.num_sgd_iter, R // MB), (shuffle, R, perms.shape)
    assert cols["idx"].dtype == torch.int32 and tuple(cols["st"].shape) == (R, 4, 23) and tuple(cols["adj"].shape) == (R, 4, 4)
    CALLS.append(("sgd_phase", R))
    cfg_o = O.PPOConfig(num_sgd_iter=self.cfg.num_sgd_iter, sgd_minibatch_size=MB)
    fwd = lambda th, obs: O.graphnet_forward(th, obs[0], obs[1], obs[2], 2 * self.A)      # noqa: E731

    class _Obs:
        def __getitem__(self, sl):
            return (cols["idx"][sl], cols["st"][sl], cols["adj"][sl])
    ob = {"obs": _Obs(), "actions": cols["act"], "old_logits": cols["logits"], "old_logp": cols["logp"],
          "vf_preds": cols["value"], "advantages": cols["adv"], "value_targets": cols["vtarg"]}
    if not hasattr(self, "_ost"):
        self._ost = O.AdamState.zeros(self.NP, torch.float32, cfg_o)
    th, st = O.sgd_loop(self.theta[0].clone(), self._ost, fwd, ob, perms.numpy(), float(self.kl_coeff_host[0]), cfg_o)
    self.theta[0] = th
    st = dict(st)
    st["cur_kl_coeff"], st["cur_lr"] = float(self.kl_coeff_host[0]), float(np.float32(self.cfg.lr))
    self._update_kl([st])
    return [st]


K.graphnet_forward, K.graphnet_act, K.gae, K.adv_standardize = graphnet_forward, graphnet_act, gae, adv_standardize
L.GraphNetLearner._sgd_phase = sgd_phase

import tests.test_gpu_graph_policy as T  # noqa: E402

for step in ("tc", "three-kernel"):
    CALLS.clear()
    T.test_graph_policy_group_serves_the_rllib_calls(step)
    # compute_actions x 2 = one fused call each; StandardizeFields over all 520 rows BEFORE the 512-row SGD phase (twice:
    # the second group of the determinism check)
    assert CALLS == ["graphnet_act", "graphnet_act"] + [("adv_standardize", 520), ("sgd_phase", 512)] * 2, CALLS
    print(step, "ok")

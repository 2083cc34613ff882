"""Float64 ground truth (and float32 twin) of one learner iteration of the leg-coupled policy of SharedDecentralLegID,
assembled from the oracle's pieces: filter -> forward -> LegCoupling -> DiagGaussian sample + logp -> bootstrap -> GAE ->
standardise -> [shuffle] -> the oracle's own `sgd_loop` (clip + TF1 Adam over all NP + 8 parameters) -> KL update.

The node id travels through `sgd_loop` as column 0 of the observation rows, so the oracle's minibatch slicing and
shuffling move it with its row and `sgd_minibatch_step` differentiates the coupled loss w.r.t. the table as well."""
import numpy as np
import torch

import oracle.ddrl_oracle as O


def coupled_forward(th, xx, NP: int):
    """xx [R, 1 + D] = (node id, observation) -> coupled logits [R, 4], value [R]."""
    lg, v = O.fcnet_forward(th[:NP], xx[:, 1:].contiguous(), 4)
    return O.leg_coupling(lg, xx[:, 0].long(), th[NP:].reshape(4, 2)), v


def coupled_learner_iteration(ps: O.PolicyState, raw_obs, boot_obs, rewards, dones, eps, shuffle, perms, cfg,
                              dtype=torch.float64):
    """ps.theta [NP + 8]; raw_obs [T, C, D] with env-major leg columns (node id of column c = c % 4), boot_obs [C, D],
    rewards [T, C], dones [T, C], eps [T, C, 2], shuffle [T*C] or None, perms [E, nb].  Updates ps, returns the columns."""
    T, C, D = raw_obs.shape
    NP = ps.theta.numel() - 8
    node = torch.from_numpy((np.arange(T * C) % C % 4).astype(np.int64))
    obs = ps.filt(raw_obs.reshape(T * C, D))
    bobs = ps.filt(boot_obs, update=False)
    x = torch.from_numpy(obs.astype(np.float32)).to(dtype)
    xb = torch.from_numpy(bobs.astype(np.float32)).to(dtype)
    xx = torch.cat([node.to(dtype)[:, None], x], dim=1)
    with torch.no_grad():
        logits, value = coupled_forward(ps.theta, xx, NP)
        act = O.dg_sample(logits, torch.from_numpy(eps.reshape(T * C, -1)).to(dtype))
        logp = O.dg_logp(logits, act)
        _, vboot = O.fcnet_forward(ps.theta[:NP], xb, 4)
    adv, vt = O.gae_recurrence(rewards, value.numpy().astype(np.float32).reshape(T, C), dones,
                               vboot.numpy().astype(np.float32), cfg.gamma, cfg.lambda_)
    adv_std = O.standardized(adv.reshape(-1))
    batch = {"obs": xx, "actions": act, "old_logits": logits, "old_logp": logp, "vf_preds": value,
             "advantages": torch.from_numpy(adv_std).to(dtype), "value_targets": torch.from_numpy(vt.reshape(-1)).to(dtype)}
    if shuffle is not None:
        idx = torch.from_numpy(shuffle.astype(np.int64))
        batch = {k: v[idx] for k, v in batch.items()}
    ps.theta, stats = O.sgd_loop(ps.theta, ps.adam, lambda th, z: coupled_forward(th, z, NP), batch, perms, ps.kl_coeff, cfg)
    ps.kl_coeff = O.update_kl(ps.kl_coeff, stats["kl"], cfg.kl_target)
    return {"stats": stats, "logits": logits, "value": value, "actions": act, "logp": logp, "batch": batch}

"""The benchmarked learner workload against the float64 oracle, at bench.py's shapes and with its own inputs.

bench.py times FullyDecentral (P = 4 policies, D = 19, A = 2), 4096 envs x T = 32 = 131 072 rows per policy, 10 epochs x 32
minibatches of 4096 rows: on a B200 the tensor-core learner runs G = 32 CTAs per policy with one full 128-row tile each, and
all 320 optimizer steps of an iteration in ONE persistent launch whose workspace (barrier tags, step counter, beta powers,
KL coefficient) carries over to the next iteration.  Three consecutive iterations on rollout sets 0, 1, 1 cover the eager
first call, a capture-and-replay of the preparation phase and a replay of an existing graph, as in bench.py's timed loop.

- A: filter, preparation phase, every step's loss statistics and the final state of each iteration against the float64
  trajectory.  The weights are compared by the error of the iteration's update, which separates float32 round-off from
  one wrong step out of 320 by orders of magnitude (the test checks that margin itself).
- B: every step teacher-forced at the device's own weights: gradient, clip + Adam arithmetic, statistics.
- C: the persistent launch is bit-identical to one launch per step, which carries B over to the launch bench.py times.
- D: a negative control: one repeated minibatch in one policy must be caught by A, at the right step and policy.

The checks take a `Workload` record (shapes, inputs, the launch shape they claim to test), so that
tests/test_gpu_supplementary_workloads.py runs the same checks on the other FCNet configurations bench.py times.

Measured errors of these checks on a B200: profiles/r03_bench_workload_errors.txt."""
import itertools
import os
from concurrent.futures import ThreadPoolExecutor
from dataclasses import dataclass

import numpy as np
import pytest
import torch

from bench import WORKLOAD, synth_rollout, workload_config
from tests.util import assert_grad_per_variable, scaled_err

pytestmark = pytest.mark.gpu

SMS = 148                      # the launch shapes below are those of a 148-SM B200
MODES = {"tc-fixed": dict(mode="tc", atomic_reduce=False),      # what bench.py's headline times
         "tc-atomic": dict(mode="tc", atomic_reduce=True),      # the library default (and bench.time_fcnet's)
         "fp32": dict(mode="fp32", atomic_reduce=False)}        # the FP32-parity line: one-step launches
COLS = ("obs", "act", "logits", "logp", "value", "adv", "vtarg")
STEP_STATS = ("policy_loss", "kl", "vf_loss", "entropy", "vf_explained_var")

# Final weights: error of the iteration's update against the float64 trajectory, max |theta - theta64| / max |update64|.
# Bound max(10 x the float32 torch twin, UPD_FLOOR); one wrong step out of 320 moves it by >= 1e-3.
UPD_FLOOR = 1e-4
# Adam moments after 320 steps, error relative to their scale: max(10 x twin, MV_FLOOR)
MV_FLOOR = 1e-3
# per-step loss statistics along the trajectory (A) and at the device's weights (B), in the units of
# |d| / max(1, |ref|) for policy loss / kl / entropy, |d| / |ref| for the vf loss, |d| for the explained variance
STAT_TOL_A = np.array([1e-4, 1e-4, 1e-4, 1e-4, 1e-3])
STAT_TOL_B = np.array([1e-5, 1e-5, 1e-5, 1e-5, 1e-4])


# PPO's clipped surrogate has a kink at ratio = 1 -+ clip_param: on one side a row passes its full gradient
# adv * ratio * dlogp / MB, on the other none.  For a row whose ratio lies within float32 round-off of the kink, a float32
# kernel and the float64 reference may take different sides, and for a far-tail action (dlogp/dlog_std = z^2 - 1) that
# one row moves the step's gradient by percent.  Bench's own inputs contain such a row: step 283 of policy 1 in the first
# iteration, ratio 0.7999995 (5e-7, ~9 float32 ulps, from 0.8); every float32 path takes the other side than float64 there.
# Rows within NEAR_CLIP of a boundary are therefore ambiguous: B accepts either side for them (one reference gradient per
# choice), and A compares a policy's trajectory only up to the first step with such a row (the loss statistics of that
# step included, nothing that depends on the update).  Everything else stays strict.  In the first iteration the
# next-closest rows of policies 1 and 0 are 2.9e-6 and 6.8e-6 from a boundary; every path takes the same side there.
NEAR_CLIP = 2e-6


@dataclass
class Workload:
    """One benchmarked FCNet configuration: its shapes, bench.py's inputs for it and the launch shape the checks claim to
    test.  `sets` are rollout sets on the host (bench.synth_rollout's dict), `iter_sets` the set of each of the three
    iterations, `theta0` [P, NP] the initial weights.  tc_setup / fp32_setup: what FCNetLearner._sgd_setup returns
    (MB, nb, G) in each kernel family; tc_rows: the rows each of the G CTAs of a tensor-core step holds.  control:
    (policy, step) of the repeated-minibatch control of D."""
    name: str
    P: int
    D: int
    A: int
    T: int
    C: int
    E: int
    NB: int
    MB: int
    sets: list
    iter_sets: tuple
    theta0: torch.Tensor
    tc_setup: tuple
    tc_rows: tuple
    fp32_setup: tuple
    control: tuple

    @property
    def R(self):
        return self.T * self.C

    @property
    def STEPS(self):
        return self.E * self.NB

    @property
    def VALUE_BIAS(self):
        """Flat index of value_out/bias: the last variable of the FCNet layout (11204 for D = 19, A = 2)."""
        return self.theta0.shape[1] - 1


def _headline():
    """bench.py's headline: FullyDecentral, rollout sets 0 and 1 of rank 0 (seeds 1234 + 100 s) on the host, three
    iterations on sets 0, 1, 1 (eager, capture + replay, replay), policy 2's step 200 as the control."""
    from ddrl_b200.modelv2 import fcnet_init_flat
    W = WORKLOAD
    P, D, A, T, E, NB, ENVS = W["P"], W["D"], W["A"], W["T"], W["epochs"], W["minibatches_per_epoch"], W["envs_per_gpu"]
    cfg = workload_config(ENVS, 1, NB, 2)
    R, MB = cfg["rows_per_policy_per_gpu"], cfg["sgd_minibatch_size_global"]
    C = R // T
    gen = torch.Generator().manual_seed(1234)
    theta0 = torch.stack([fcnet_init_flat(D, 2 * A, gen) for _ in range(P)])       # as bench.py
    sets = [synth_rollout(P, T, C, D, A, ENVS, NB, E, 1234 + 100 * s) for s in range(2)]
    return Workload(name="FullyDecentral", P=P, D=D, A=A, T=T, C=C, E=E, NB=NB, MB=MB, sets=sets, iter_sets=(0, 1, 1),
                    theta0=theta0, tc_setup=(4096, 32, 32), tc_rows=(128,) * 32, fp32_setup=(4096, 32, 37),
                    control=(2, 200))


def _oracle():
    import oracle.ddrl_oracle as O
    return O


def _cfg_o(w):
    return _oracle().PPOConfig(num_sgd_iter=w.E, sgd_minibatch_size=w.MB)


def _learner(w, mode, **kw):
    """FCNetLearner with bench.py's arguments, in the kernel family / reduction of `mode`."""
    from ddrl_b200.config import PPOConfig
    from ddrl_b200.learner import FCNetLearner
    return FCNetLearner(w.P, w.D, w.A, PPOConfig(num_sgd_iter=w.E, sgd_minibatch_size=w.MB), "cuda", theta=w.theta0,
                        **MODES[mode], **kw)


def cta_rows(MB, G):
    """Rows of each of the G CTAs of a tensor-core step within one minibatch: rpc = ((MB + G - 1) / G + 7) & ~7 rows per
    CTA in CTA order, the last ones ragged or empty (csrc/tc2_step_body.inc)."""
    rpc = (((MB + G - 1) // G) + 7) & ~7
    return tuple(min((bx + 1) * rpc, MB) - min(bx * rpc, MB) for bx in range(G))


def _assert_bench_shape(w, L, mode, persistent=True):
    """The launch shape this file claims to test; fails if the learner's choice drifts."""
    from ddrl_b200 import kernels as K
    MB_, nb, G = L._sgd_setup(w.R)
    assert L.sms == SMS, f"{L.sms} SMs: the launch shapes asserted here are those of the {SMS}-SM B200"
    if MODES[mode]["mode"] == "tc":
        assert K.tc_pingpong_eligible(w.D, w.A)                # the ping-pong kernel (persistent launch)
        assert (MB_, nb, G) == w.tc_setup, (MB_, nb, G)
        assert cta_rows(MB_, G) == w.tc_rows, cta_rows(MB_, G)
        assert L._persistent_steps(G) == persistent
    else:
        assert (MB_, nb, G) == w.fp32_setup, (MB_, nb, G, L.sms)
        assert not L._persistent_steps(G)
    assert L.fuse_tail and G * w.P <= L.sms                    # reduce + clip + Adam inside the train kernel
    assert L.atomic_reduce == MODES[mode]["atomic_reduce"], "partial-gradient reduction is not the intended one (DDRL_FIXED_ORDER?)"


def _to_dev(r):
    return {k: v.to("cuda") for k, v in r.items()}


def _learn(L, r):
    return L.learn_on_rollout(r["raw"], r["boot"], r["rewards"], r["dones"], r["eps"], r["perms"], r["shuffle"])


def _clip_branch(logits, act, old_logp, adv, cfg):
    """Per row: ratio, whether the clipped surrogate passes the row's gradient (ratio inside [1 - c, 1 + c] or the unclipped
    term is the smaller one, as torch.minimum / torch.clamp and csrc/ppo_loss.cuh decide) and whether the ratio lies within
    NEAR_CLIP of a boundary."""
    O = _oracle()
    ratio = torch.exp(O.dg_logp(logits, act) - old_logp)
    lo, hi = 1.0 - cfg.clip_param, 1.0 + cfg.clip_param
    flows = ((ratio >= lo) & (ratio <= hi)) | (adv * ratio <= adv * ratio.clamp(lo, hi))
    near = torch.minimum((ratio - lo).abs(), (ratio - hi).abs()) < NEAR_CLIP
    return ratio, flows, near


# ---- the float64 oracle trajectory --------------------------------------------------------------------------------------
def _oracle_policy(w, p, sets):
    """Three learner iterations of policy p (w.iter_sets) in float64, step by step, and in float32 (the torch twin).
    -> one record per iteration; `cut` = the first step of the iteration with a row within NEAR_CLIP of the clip kink or
    a row on which the twin takes the other side of the kink than float64 (`fork`: that step and the float64 distance of
    such rows from the kink), `after_cut` = an earlier iteration had one."""
    O = _oracle()
    cfg = _cfg_o(w)
    P, D, A, T, C, E, R, MB = w.P, w.D, w.A, w.T, w.C, w.E, w.R, w.MB
    theta0 = w.theta0[p]
    filt = O.MeanStdFilter((D,), clip=None)      # the learner's filter_clip = 0: RLlib's MeanStdFilter has clip=None
    state = {dt: [theta0.to(dt), O.AdamState.zeros(theta0.numel(), dt, cfg), cfg.kl_coeff] for dt in (torch.float64, torch.float32)}
    fwd = lambda th, x: O.fcnet_forward(th, x, 2 * A)
    out = []
    forked = False      # why this trajectory is one of several valid ones from here on (a row at the clip kink, ...)
    for s in w.iter_sets:
        r = sets[s]
        obs = filt(r["raw"][p].reshape(R, D))                  # pushes every row, then normalises
        bobs = filt(r["boot"][p], update=False)
        rec = {"filt": (filt.rs.n, filt.rs._M.copy(), filt.rs._S.copy())}
        sides, dist = {}, []      # per step: the rows' side of the kink in each dtype, their float64 distance from it
        for dt in (torch.float64, torch.float32):
            theta, adam, klc = state[dt]
            x = torch.from_numpy(obs.astype(np.float32)).to(dt)
            with torch.no_grad():
                logits, value = fwd(theta, x)
                act = O.dg_sample(logits, torch.from_numpy(r["eps"][p].reshape(R, A)).to(dt))
                logp = O.dg_logp(logits, act)
                _, vboot = fwd(theta, torch.from_numpy(bobs.astype(np.float32)).to(dt))
            adv, vt = O.gae_recurrence(r["rewards"][p], value.numpy().astype(np.float32).reshape(T, C), r["dones"],
                                       vboot.numpy().astype(np.float32), cfg.gamma, cfg.lambda_)
            adv_std = O.standardized(adv.reshape(-1))
            batch = {"obs": x, "actions": act, "old_logits": logits, "old_logp": logp, "vf_preds": value,
                     "advantages": torch.from_numpy(adv_std).to(dt), "value_targets": torch.from_numpy(vt.reshape(-1)).to(dt)}
            idx = torch.from_numpy(r["shuffle"][p].astype(np.int64))
            batch = {k: v[idx] for k, v in batch.items()}
            theta_first = theta_last = None
            steps, cut, sides[dt] = [], None, []
            for e in range(E):
                last = {k: [] for k in O.STAT_KEYS}
                for mb in r["perms"][p, e]:
                    rows = slice(int(mb) * MB, (int(mb) + 1) * MB)
                    if dt == torch.float64:      # O.sgd_minibatch_step + the rows near the clip kink
                        theta_last = theta
                        theta_first = theta if theta_first is None else theta_first
                        th = theta.clone().requires_grad_(True)
                        lg, v = fwd(th, batch["obs"][rows])
                        loss, st = O.ppo_loss_from_outputs(lg, v, *(batch[k][rows] for k in (
                            "actions", "old_logits", "old_logp", "vf_preds", "advantages", "value_targets")), klc, cfg)
                        (g,) = torch.autograd.grad(loss, th)
                        ratio, flows, near = _clip_branch(lg.detach(), batch["actions"][rows], batch["old_logp"][rows],
                                                          batch["advantages"][rows], cfg)
                        if cut is None and bool(near.any()):
                            cut = len(steps)
                        sides[dt].append(flows.numpy())
                        dist.append(torch.minimum((ratio - 1.0 + cfg.clip_param).abs(), (ratio - 1.0 - cfg.clip_param).abs()).numpy())
                        theta = O.adam_tf1_step(theta, O.clip_by_global_norm(g, cfg.grad_clip)[0], adam, cfg)
                        st = {k: float(x.detach()) for k, x in st.items()}
                    else:
                        with torch.no_grad():
                            lg = fwd(theta, batch["obs"][rows])[0]
                        sides[dt].append(_clip_branch(lg, batch["actions"][rows], batch["old_logp"][rows],
                                                      batch["advantages"][rows], cfg)[1].numpy())
                        theta, st, _, _ = O.sgd_minibatch_step(theta, adam, fwd, batch, rows, klc, cfg)
                    steps.append([st[k] for k in STEP_STATS])
                    for k in O.STAT_KEYS:
                        last[k].append(st[k])
            stats = {k: float(np.mean(np.asarray(v, dtype=np.float32))) for k, v in last.items()}     # as O.sgd_loop
            klc = O.update_kl(klc, stats["kl"], cfg.kl_target)
            state[dt] = [theta, adam, klc]
            if dt == torch.float64:
                rec.update(obs=obs, logits=logits.numpy(), value=value.numpy(), act=act.numpy(), logp=logp.numpy(),
                           adv=adv_std, vtarg=vt.reshape(-1), step_stats=np.array(steps), theta_first=theta_first.numpy(),
                           theta_last=theta_last.numpy(), theta=theta.numpy(), m=adam.m.numpy().copy(),
                           v=adam.v.numpy().copy(), beta_pow=(adam.beta1_power, adam.beta2_power), kl_coeff=klc, stats=stats,
                           cut=cut, after_cut=forked)
            else:
                rec.update(twin_theta=theta.numpy().astype(np.float64), twin_m=adam.m.numpy().astype(np.float64),
                           twin_v=adam.v.numpy().astype(np.float64))
        # a row far enough from the kink for NEAR_CLIP, on which float32 round-off still took the other side
        fork = next((i for i, (a, b) in enumerate(zip(sides[torch.float64], sides[torch.float32])) if (a != b).any()), None)
        if fork is not None:
            flip = sides[torch.float64][fork] != sides[torch.float32][fork]
            rec["fork"] = (fork, float(dist[fork][flip].min()))
            rec["cut"] = fork if rec["cut"] is None else min(rec["cut"], fork)
        # the end state resolves one wrong step only if float32 round-off alone (the twin) leaves it more than 10x closer
        # to float64 than the trajectory without its last step; where it does not (Adam amplifies round-off on
        # near-zero gradients), a float32 trajectory of this policy is one of many valid ones from here on
        rec["resolved"] = _update_err(rec["theta_last"], rec) > 10.0 * max(10.0 * _update_err(rec["twin_theta"], rec), UPD_FLOOR)
        forked = forked or ("reached the clip kink" if rec["cut"] is not None else
                            "left the float32 trajectories unresolved" if not rec["resolved"] else False)
        out.append(rec)
    return out


def oracle_trajectory(w):
    """-> [iteration][policy] records of the float64 trajectory (+ the twin's final state).  The policies are independent and
    run on P host threads, as bench.CpuLearner does."""
    sets = [{k: v.numpy() for k, v in r.items()} for r in w.sets]
    threads = torch.get_num_threads()
    torch.set_num_threads(max(1, (os.cpu_count() or 1) // w.P))
    try:
        with ThreadPoolExecutor(w.P) as ex:
            per_policy = list(ex.map(lambda p: _oracle_policy(w, p, sets), range(w.P)))
    finally:
        torch.set_num_threads(threads)
    return [[per_policy[p][i] for p in range(w.P)] for i in range(len(w.iter_sets))]


@pytest.fixture(scope="module")
def headline():
    return _headline()


@pytest.fixture(scope="module")
def oracle(headline):
    return oracle_trajectory(headline)


# ---- comparisons ----------------------------------------------------------------------------------------------------------
def _device_step_stats(ss, MB):
    """step_stats [steps, P, 8] float64 sums over the MB rows of a step -> [steps, P, 5] in STEP_STATS order."""
    s = np.asarray(ss, dtype=np.float64) / MB
    ev = np.maximum(-1.0, 1.0 - (s[..., 7] - s[..., 6] ** 2) / (s[..., 5] - s[..., 4] ** 2))
    return np.stack([s[..., 0], s[..., 1], s[..., 2], s[..., 3], ev], axis=-1)


def _stat_ratio(dev, ref, tol):
    """Per-stat error over its tolerance, max over the stats (<= 1 passes)."""
    d = np.abs(dev - ref)
    den = np.maximum(1.0, np.abs(ref))
    den[..., 2] = np.abs(ref[..., 2])
    den[..., 4] = 1.0
    return (d / den / tol).max(axis=-1)


def _update_err(theta, ref):
    """max |theta - theta64| over the size of the float64 update of the iteration."""
    upd = ref["theta"] - ref["theta_first"]
    return float(np.abs(np.asarray(theta, dtype=np.float64) - ref["theta"]).max() / np.abs(upd).max())


def _beta_chain(steps):
    b = np.float32(0.9), np.float32(0.999)
    out = list(b)
    for _ in range(steps):
        out = [np.float32(out[0] * b[0]), np.float32(out[1] * b[1])]
    return out


def compared_steps(w, ref):
    """Steps of an iteration whose loss statistics A compares for one policy: all, up to the first step with a row at
    the clip kink, or none after an earlier iteration had one."""
    return 0 if ref["after_cut"] else w.STEPS if ref["cut"] is None else ref["cut"] + 1


def _compare(w, L, stats, refs, it, tag):
    """One learn_on_rollout result against the oracle's iteration `it` -> (failures [(policy, message)], first off step or
    None, per-policy measurements).  Prints one line per policy with the measured errors.  A policy whose reference
    trajectory reached a row at the clip kink (NEAR_CLIP) is compared up to that step only; the filter, the normalised
    observations, the beta powers and tc_status do not depend on the weights and are checked always."""
    P, R = w.P, w.R
    fails = []
    bufs = L._bufs
    ss = _device_step_stats(bufs["step_stats"].cpu().numpy(), w.MB)
    ratio = np.stack([_stat_ratio(ss[:, p], refs[p]["step_stats"], STAT_TOL_A) for p in range(P)], axis=1)    # [steps, P]
    for p in range(P):
        if refs[p]["after_cut"]:
            ratio[:, p] = 0.0
        elif refs[p]["cut"] is not None:
            ratio[refs[p]["cut"] + 1:, p] = 0.0
    bad = np.argwhere(ratio > 1.0)
    first = tuple(int(x) for x in bad[0]) if len(bad) else None
    if first is not None:
        fails.append((first[1], f"it {it}: step statistics first off at step {first[0]}, policy {first[1]} "
                                f"(error / tolerance {ratio[first]:.3g})"))
    beta = _beta_chain(w.STEPS * (it + 1))
    theta, m, v = L.theta.cpu().numpy(), L.m.cpu().numpy(), L.v.cpu().numpy()
    bp, klc = L.beta_pow.cpu().numpy(), L.kl_coeff.cpu().numpy()
    meas = []
    for p in range(P):
        ref = refs[p]

        def check(ok, msg):
            if not ok:
                fails.append((p, f"it {it} policy {p}: {msg}"))
        n, M, S = ref["filt"]
        check(int(L.filt_n[p]) == n == R * (it + 1), f"filter count {int(L.filt_n[p])} != {n}")
        check(np.allclose(L.filt_M[p].cpu().numpy(), M, rtol=1e-12, atol=1e-12), "filter mean")
        check(np.allclose(L.filt_S[p].cpu().numpy(), S, rtol=1e-11, atol=0.0), "filter M2")
        e = scaled_err(bufs["obs"][p].cpu().numpy(), ref["obs"])
        check(e < 1e-6, f"obs error {e:.3g} >= 1e-6")
        check(bp[p, 0] == beta[0] and bp[p, 1] == beta[1], f"beta powers {bp[p]} != float32 chain {beta}")
        if ref["after_cut"]:
            meas.append(None)
            print(f"[A {tag} it={it} p={p}] weight-dependent checks skipped: an earlier iteration {ref['after_cut']}")
            continue
        for name, tol in (("logits", 1e-5), ("value", 1e-5), ("act", 1e-5), ("logp", 1e-5), ("vtarg", 1e-5), ("adv", 2e-5)):
            e = scaled_err(bufs[name][p].cpu().numpy(), ref[name])
            check(e < tol, f"{name} error {e:.3g} >= {tol}")
        if ref["cut"] is not None:
            meas.append(None)
            print(f"[A {tag} it={it} p={p}] step statistics compared up to step {ref['cut']} (a row at the clip kink), "
                  f"step_stats_err/tol={ratio[:, p].max():.3g}")
            continue
        if not ref["resolved"]:
            meas.append(None)
            print(f"[A {tag} it={it} p={p}] step statistics compared over all steps, step_stats_err/tol="
                  f"{ratio[:, p].max():.3g}; end state not compared: the float32 twin alone is "
                  f"{_update_err(ref['twin_theta'], ref):.3g} of the update from float64, the trajectory without its last "
                  f"step {_update_err(ref['theta_last'], ref):.3g}")
            continue
        upd = _update_err(theta[p], ref)
        twin = _update_err(ref["twin_theta"], ref)
        bound = max(10.0 * twin, UPD_FLOOR)
        guard = _update_err(ref["theta_last"], ref)          # the float64 trajectory without its last step
        check(guard > 10.0 * bound, f"last-step guard {guard:.3g} is not 10x above the bound {bound:.3g}")
        check(upd < bound, f"update error {upd:.3g} >= {bound:.3g} (twin {twin:.3g})")
        em, ev_ = scaled_err(m[p], ref["m"]), scaled_err(v[p], ref["v"])
        em_t, ev_t = scaled_err(ref["twin_m"], ref["m"]), scaled_err(ref["twin_v"], ref["v"])
        check(em < max(10.0 * em_t, MV_FLOOR), f"adam m error {em:.3g} (twin {em_t:.3g})")
        check(ev_ < max(10.0 * ev_t, MV_FLOOR), f"adam v error {ev_:.3g} (twin {ev_t:.3g})")
        check(L.kl_coeff_host[p] == ref["kl_coeff"] and klc[p] == np.float32(ref["kl_coeff"]),
              f"kl coefficient {L.kl_coeff_host[p]} / {klc[p]} != {ref['kl_coeff']}")
        for k, rv in ref["stats"].items():
            check(abs(stats[p][k] - rv) < 1e-4 * max(1.0, abs(rv)), f"returned {k} {stats[p][k]} != {rv}")
        meas.append(dict(upd=upd, twin=twin, bound=bound, guard=guard, stat=float(ratio[:, p].max()), m=em, v=ev_))
        print(f"[A {tag} it={it} p={p}] update_err={upd:.3g} twin={twin:.3g} bound={bound:.3g} guard={guard:.3g} "
              f"step_stats_err/tol={ratio[:, p].max():.3g} m_err={em:.3g} (twin {em_t:.3g}) v_err={ev_:.3g} (twin {ev_t:.3g})")
    if int(L.tc_status) != 0:
        fails.append((-1, f"it {it}: tc_status {int(L.tc_status)}"))
    return fails, first, meas


def check_iterations(w, mode, oracle, tag):
    """A: the three iterations of w.iter_sets on a bench-style learner against the float64 trajectory -> the failures."""
    sets = [_to_dev(r) for r in w.sets]
    L = _learner(w, mode)
    _assert_bench_shape(w, L, mode)
    fails = []
    for it, s in enumerate(w.iter_sets):
        stats = _learn(L, sets[s])
        torch.cuda.synchronize()
        fails += [msg for _, msg in _compare(w, L, stats, oracle[it], it, tag)[0]]
    assert L._prep_graphs is not None and len(L._prep_graphs) == len(set(w.iter_sets[1:])), getattr(L, "graph_error", None)
    if mode == "fp32":
        assert L._graph is not None, getattr(L, "graph_error", None)      # graph-captured one-step launches
    return fails


@pytest.mark.parametrize("mode", list(MODES))
def test_bench_workload_iterations_match_oracle(mode, headline, oracle):
    """Three bench-shaped iterations (sets 0, 1, 1): filter, preparation phase, the 320 steps' loss statistics and the
    final weights / Adam state / beta powers / KL coefficient / returned stats of each, against the float64 oracle."""
    fails = check_iterations(headline, mode, oracle, mode)
    assert not fails, "\n".join(fails)


def _loss_grad(w, theta, cols, p, rows, klc, cfg, dtype):
    """autograd of the mean PPO loss over cols[*][p][rows] at theta -> (reference gradients, [5] stats in STEP_STATS
    order, max |v|).  The first gradient is torch's; float64 adds one per non-empty subset of the rows within NEAR_CLIP of
    the clip kink, with those rows on the other side of it."""
    O = _oracle()
    th = torch.from_numpy(theta).to(dtype).requires_grad_(True)
    c = {k: cols[k][p, rows].to(dtype) for k in COLS}
    lg, v = O.fcnet_forward(th, c["obs"], 2 * w.A)
    loss, st = O.ppo_loss_from_outputs(lg, v, c["act"], c["logits"], c["logp"], c["value"], c["adv"], c["vtarg"], klc, cfg)
    near_rows = []
    if dtype == torch.float64:
        ratio, flows, near = _clip_branch(lg, c["act"], c["logp"], c["adv"], cfg)
        near_rows = near.nonzero().reshape(-1).tolist()
        assert len(near_rows) <= 3, f"{len(near_rows)} rows at the clip kink"
    (g,) = torch.autograd.grad(loss, th, retain_graph=bool(near_rows))
    deltas = []
    for i, r in enumerate(near_rows):
        # the loss holds -mean(surr): a row on the gradient-passing side contributes -d(adv * ratio) / MB
        (d,) = torch.autograd.grad(c["adv"][r] * ratio[r], th, retain_graph=i + 1 < len(near_rows))
        deltas.append((d if bool(flows[r]) else -d) / ratio.numel())
    refs = [g + sum(sub, torch.zeros_like(g)) for k in range(len(deltas) + 1) for sub in itertools.combinations(deltas, k)]
    return ([x.numpy().astype(np.float64) for x in refs], np.array([float(st[k].detach()) for k in STEP_STATS]),
            float(v.detach().abs().max()))


def grad_check(w, mode, grad, th0, cols, p, rows, klc, cfg):
    """B's gradient rule for one policy's step -> (scaled error, value-bias error over 1e-5 max|v|, kink rows present,
    failure message or None).  Rows at the clip kink: the side the kernel took, and the twin's round-off around the side
    it took."""
    gtol = 5e-5 if MODES[mode]["mode"] == "tc" else 1e-5
    shapes = [shp for _, shp in _oracle().fcnet_shapes(w.D, 2 * w.A)]
    refs, st64, vmax = _loss_grad(w, th0, cols, p, rows, klc, cfg, torch.float64)
    (g32,), _, _ = _loss_grad(w, th0, cols, p, rows, klc, cfg, torch.float32)
    g64 = min(refs, key=lambda x: scaled_err(grad, x))
    twin = g32 - min(refs, key=lambda x: scaled_err(g32, x)) + g64
    e = scaled_err(grad, g64)
    msg = f"gradient error {e:.3g} >= {gtol}" if e >= gtol else None
    # value_out/bias = vf_loss_coeff * 2 * mean(v - R): its error is the mean error of the step's value forward,
    # which the tensor-core path holds to 1e-5 of the value's scale (not a cancelling sum that round-off averages)
    vb_allow = 2.0 * cfg.vf_loss_coeff * 1e-5 * vmax
    allow = {w.VALUE_BIAS: vb_allow} if MODES[mode]["mode"] == "tc" else None
    vb = abs(grad[w.VALUE_BIAS] - g64[w.VALUE_BIAS]) / vb_allow
    try:
        assert_grad_per_variable(grad, g64, twin, shapes, gtol, allow=allow)
    except AssertionError as exc:
        msg = f"{msg + '; ' if msg else ''}gradient per variable: {exc}"
    return e, vb, len(refs) > 1, msg, st64


def _step_rows(w, perms, p, s):
    mb = int(perms[p, s // w.NB, s % w.NB])
    return slice(mb * w.MB, (mb + 1) * w.MB)


def check_every_step(w, mode, tag):
    """B: the first iteration (set w.iter_sets[0]), one eager launch per step (fused tail at the bench's G), teacher-forced:
    at every step the device's reduced gradient against float64 autograd at the device's weights on the device's own
    shuffled columns, the device's clip + Adam against float64 arithmetic from its own gradient and state, and the step's
    statistics.  Prints the worst errors per policy -> the failures (at most 20)."""
    cfg = _cfg_o(w)
    P = w.P
    f32 = lambda x: float(np.float32(x))
    b1, b2, lr, eps, clip = (f32(x) for x in (cfg.beta1, cfg.beta2, cfg.lr, cfg.adam_eps, cfg.grad_clip))
    gtol = 5e-5 if MODES[mode]["mode"] == "tc" else 1e-5
    r = w.sets[w.iter_sets[0]]
    perms = r["perms"].numpy()
    L = _learner(w, mode, persistent=False, use_graph=False)
    _assert_bench_shape(w, L, mode, persistent=False)
    orig = L._sgd_step
    ctx = {"step": 0, "cols": None}
    fails = []
    worst = {k: np.zeros(P) for k in ("grad", "m", "v", "theta", "gnorm", "stat", "vbias", "kink")}

    def fail(s, p, msg):
        if len(fails) < 20:
            fails.append(f"step {s} policy {p}: {msg}")

    def step(b, MB_, G, hyper, src, nsteps=1):
        s = ctx["step"]
        ctx["step"] += 1
        torch.cuda.synchronize()
        th0, m0, v0, bp0, klc = (t.cpu().numpy().astype(np.float64) for t in (L.theta, L.m, L.v, L.beta_pow, L.kl_coeff))
        orig(b, MB_, G, hyper, src, nsteps)
        torch.cuda.synchronize()
        grad, gn, th1, m1, v1 = (t.cpu().numpy().astype(np.float64) for t in (L.grad, L.gnorm, L.theta, L.m, L.v))
        bp1 = L.beta_pow.cpu().numpy()
        ss = _device_step_stats(b["step_stats"][s:s + 1].cpu().numpy(), w.MB)[0]
        if ctx["cols"] is None:
            ctx["cols"] = {k: src[k].cpu() for k in COLS}

        def one(p):
            rows = _step_rows(w, perms, p, s)
            # 1. gradient
            e, vb, kink, msg, st64 = grad_check(w, mode, grad[p], th0[p], ctx["cols"], p, rows, klc[p], cfg)
            worst["kink"][p] += kink
            worst["grad"][p] = max(worst["grad"][p], e)
            worst["vbias"][p] = max(worst["vbias"][p], vb)
            if msg is not None:
                fail(s, p, msg)
            # 2. global-norm clip + TF1 Adam in float64 from the device's own gradient and state
            norm = float(np.sqrt((grad[p] ** 2).sum()))
            gc = grad[p] * (clip * min(1.0 / norm, 1.0 / clip))
            lr_t = lr * np.sqrt(1.0 - bp0[p, 1]) / (1.0 - bp0[p, 0])
            m = m0[p] + (gc - m0[p]) * (1.0 - b1)
            v = v0[p] + (gc * gc - v0[p]) * (1.0 - b2)
            th = th0[p] - (m * lr_t) / (np.sqrt(v) + eps)
            errs = dict(gnorm=abs(gn[p] - norm) / norm, m=scaled_err(m1[p], m), v=scaled_err(v1[p], v),
                        theta=float((np.abs(th1[p] - th) / (5e-7 * np.abs(th) + 1e-9)).max()))    # <= 1: rtol 5e-7, atol 1e-9
            for k, x in errs.items():
                worst[k][p] = max(worst[k][p], x)
                if x >= (1.0 if k == "theta" else 1e-6):
                    fail(s, p, f"tail arithmetic: {k} error {x:.3g}")
            if not (bp1[p, 0] == np.float32(np.float32(bp0[p, 0]) * np.float32(b1))
                    and bp1[p, 1] == np.float32(np.float32(bp0[p, 1]) * np.float32(b2))):
                fail(s, p, f"beta powers {bp0[p]} -> {bp1[p]}")
            # 3. loss statistics at the device's weights
            x = float(_stat_ratio(ss[p], st64, STAT_TOL_B))
            worst["stat"][p] = max(worst["stat"][p], x)
            if x > 1.0:
                fail(s, p, f"step statistics error / tolerance {x:.3g}: {ss[p]} vs {st64}")

        list(pool.map(one, range(P)))

    L._sgd_step = step
    threads = torch.get_num_threads()
    torch.set_num_threads(max(1, (os.cpu_count() or 1) // P))
    try:
        with ThreadPoolExecutor(P) as pool:      # the float64 autograd of the P policies side by side
            _learn(L, _to_dev(r))
    finally:
        torch.set_num_threads(threads)
    torch.cuda.synchronize()
    assert ctx["step"] == w.STEPS
    for p in range(P):
        print(f"[B {tag} it=0 p={p}] grad_err={worst['grad'][p]:.3g} (tol {gtol}) gnorm_err={worst['gnorm'][p]:.3g} "
              f"m_err={worst['m'][p]:.3g} v_err={worst['v'][p]:.3g} theta_err/tol={worst['theta'][p]:.3g} "
              f"step_stats_err/tol={worst['stat'][p]:.3g} value_bias_err/(1e-5 max|v|)={worst['vbias'][p]:.3g} "
              f"steps_with_a_row_at_the_clip_kink={int(worst['kink'][p])}")
    return fails


@pytest.mark.parametrize("mode", list(MODES))
def test_every_step_matches_oracle_at_device_weights(mode, headline):
    """First iteration, one eager launch per step (fused tail at the bench's G), teacher-forced: at every step the
    device's reduced gradient against float64 autograd at the device's weights on the device's own shuffled columns, the
    device's clip + Adam against float64 arithmetic from its own gradient and state, and the step's statistics."""
    fails = check_every_step(headline, mode, mode)
    assert not fails, "\n".join(fails)


def check_persistent_equals_one_step(w):
    """C: with the fixed-order reduction, the bench-style learner (ONE persistent launch per iteration, graph-replayed
    preparation) and the learner of B (one eager launch per step) leave bit-identical state after each iteration."""
    sets = [_to_dev(r) for r in w.sets]
    La = _learner(w, "tc-fixed")
    Lb = _learner(w, "tc-fixed", persistent=False, use_graph=False)
    _assert_bench_shape(w, La, "tc-fixed")
    _assert_bench_shape(w, Lb, "tc-fixed", persistent=False)
    for it, s in enumerate(w.iter_sets):
        sa, sb = _learn(La, sets[s]), _learn(Lb, sets[s])
        torch.cuda.synchronize()
        a, b = La._bufs["step_stats"], Lb._bufs["step_stats"]
        diff = (a != b).reshape(w.STEPS, -1).any(dim=1).nonzero()
        assert len(diff) == 0, f"iteration {it}: step statistics first differ at step {int(diff[0])}"
        for name in ("theta", "m", "v", "beta_pow", "kl_coeff", "filt_n", "filt_M", "filt_S"):
            assert torch.equal(getattr(La, name), getattr(Lb, name)), (it, name)
        assert sa == sb, it


def test_persistent_launch_equals_one_step_launches(headline):
    """Fixed-order reduction: the bench-style learner (ONE persistent launch of 320 steps, graph-replayed preparation) and
    the learner of B (one eager launch per step) leave bit-identical state after each of three iterations."""
    check_persistent_equals_one_step(headline)


def check_repeated_minibatch(w, oracle, tag):
    """D: in the first iteration, policy q's step s (w.control) repeats the minibatch of step s - 1 of the same epoch.
    Against the unmodified oracle, A must flag step s of policy q first and pass the other policies; if q's reference
    trajectory is compared to its end, q's final weights must be off by more than 10x the bound."""
    q, target = w.control
    cut = oracle[0][q]["cut"]
    assert cut is None or cut > target, f"policy {q}'s reference reaches the clip kink at step {cut}"
    e, i = divmod(target, w.NB)
    r = dict(w.sets[w.iter_sets[0]])
    perms = r["perms"].clone()
    assert i > 0 and perms[q, e, i] != perms[q, e, i - 1]
    perms[q, e, i] = perms[q, e, i - 1]
    r["perms"] = perms
    L = _learner(w, "tc-fixed")
    _assert_bench_shape(w, L, "tc-fixed")
    stats = _learn(L, _to_dev(r))
    torch.cuda.synchronize()
    fails, first, meas = _compare(w, L, stats, oracle[0], 0, tag)
    assert first == (target, q), first
    if cut is None:
        assert meas[q]["upd"] > 10.0 * meas[q]["bound"], meas[q]
    assert not [msg for p, msg in fails if p != q], fails


def test_one_wrong_minibatch_is_caught(headline, oracle):
    """Negative control at the bench shape, valid inputs: policy 2's step 200 (epoch 6, position 8) repeats the minibatch of
    step 199.  Against the unmodified oracle, A's checks must flag step 200 of policy 2 first and policy 2's final weights,
    and pass the other policies.  (Policy 2: its reference trajectory has no row at the clip kink in this iteration, so
    the whole trajectory is compared; the unfaulted learner passes the same checks in the iterations test.)"""
    assert headline.control == (2, 200) and oracle[0][2]["cut"] is None
    check_repeated_minibatch(headline, oracle, "fault")

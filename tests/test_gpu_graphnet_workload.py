"""The benchmarked GraphNet workload against the float64 oracle, at bench.py's launch shape and with its own inputs.

bench.py's second workload (`time_graphnet`: `--workload graphnet`, the `C4_shared_GraphNet` supplementary line) trains the
shared GraphNet policy on 4096 envs x 4 legs x T = 32 = 524 288 rows, 32 minibatches of 16 384 rows, E = 10 epochs.  On a
148-SM B200 `GraphNetLearner` launches Gn = 74 CTAs per net (148 in all) and runs all E x 32 steps in ONE persistent launch
of `graphnet_train_tc_kernel` (csrc/graphnet_tc.cu).  Each CTA gets rpc = ((MB + Gn - 1) / Gn + 7) & ~7 = 224 rows of a
minibatch: CTAs 0..72 walk four tiles (64, 64, 64, 32 rows), accumulating the MPNN / head weight gradients in TMEM and the
encoder gradients in registers across them under ONE gradient scale taken from the first tile; CTA 73 holds the last 32
rows in one ragged tile.  The minibatch order crosses epoch boundaries inside the launch, and the tail's barrier epoch,
the beta powers and the KL coefficient carry over from one iteration to the next.

The inputs are bench.py's own: `bench.time_graphnet` runs once per E with `GraphNetLearner.learn_on_rollout` wrapped,
which records the weights and every argument before calling through.

- A: two consecutive iterations at E = 2 (64 steps per launch), tensor-core and three-kernel step, against one float64
  trajectory and its float32 torch twin: the preparation phase, every step's loss statistics, and the weights, Adam state,
  beta powers, KL coefficient and returned statistics after each iteration.
- B: the 320 steps of the E = 10 iteration as 320 single-step launches of the same kernel on the learner's own buffers;
  at nine sampled steps (first, last, epoch boundaries) the reduced gradient against float64 autograd at the device's
  weights, the clip + TF1 Adam arithmetic, and the step's statistics.
- C: the persistent 320-step launch is bit-identical to B's single-step launches, and to itself when repeated.
- D: negative controls (a repeated minibatch, one lost ragged CTA) that the checks must catch, and a stress check of the
  first-tile gradient scale that must either pass or raise the kernel's overflow flag.

Measured errors of these checks on a B200: profiles/r08_graphnet_workload_errors.txt."""
import contextlib
import itertools
import os
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest
import torch

from tests.test_gpu_bench_workload import (MV_FLOOR, STAT_TOL_A, STAT_TOL_B, STEP_STATS, UPD_FLOOR, _beta_chain,
                                           _clip_branch, _stat_ratio)
from tests.util import assert_grad_per_variable, scaled_err

pytestmark = pytest.mark.gpu

A, T, ENVS, NB = 2, 32, 4096, 32                 # bench.time_graphnet's shape
C = ENVS * 4
R = T * C
MB = R // NB
SMS, GN = 148, 74                                # a B200: Gn = sms // 2 CTAs per net
E_A, E_B = 2, 10                                 # A: --gn-epochs 2 (64 steps per launch); B, C: the bench's E = 10
SAMPLED = (0, 1, 31, 32, 63, 64, 159, 288, 319)  # B: first / last steps and epoch boundaries
CONTROL_STEP = 159                               # D: the step whose launch is repeated with modified advantages
RAGGED_CTA = GN - 1                              # holds the minibatch's last 32 rows
STRESS_CTA = 0
CHUNK = 16384                                    # rows per oracle forward call of the preparation phase
COLS = ("act", "logits", "logp", "value", "adv", "vtarg")
TC_GRAD_TOL = 5e-5       # the tensor-core step's gradient tolerance (fp16 hi/lo split operands), as in test_gpu_graphnet_train
FWD_TOL = 1e-5           # forward outputs (logits, value) relative to their scale: the FP32 forward and the tc step alike
PREP_TOL = {"logits": FWD_TOL, "value": FWD_TOL, "vboot": FWD_TOL, "act": FWD_TOL, "logp": FWD_TOL, "vtarg": FWD_TOL,
            "gae_adv": 2e-5, "adv": 2e-5, "moments": 2e-5}


def _oracle():
    import oracle.ddrl_oracle as O
    return O


def _cfg_o(E):
    return _oracle().PPOConfig(num_sgd_iter=E, sgd_minibatch_size=MB)


def _rpc(mb, gn):
    """Rows per CTA of one minibatch: the formula of graphnet_train_tc_kernel."""
    return (((mb + gn - 1) // gn) + 7) & ~7


def _cta_rows(mb, gn):
    """-> [(first row, rows)] of every CTA of a net within one minibatch, as the kernel splits it."""
    rpc = _rpc(mb, gn)
    out = []
    for bx in range(gn):
        r0 = min(bx * rpc, mb)
        out.append((r0, min(r0 + rpc, mb) - r0))
    return out


# ---- instrumentation ---------------------------------------------------------------------------------------------------
@contextlib.contextmanager
def _instrumented(log, keep_args=False, tc_hook=None):
    """Wraps GraphNetLearner.learn_on_rollout and the kernels it calls; appends one record per learn_on_rollout call to
    `log`: the preparation phase's outputs (forward, bootstrap forward, GAE + moments, the columns handed to the SGD phase),
    every `graphnet_train_step_tc` launch (rows, A, MB, Gn, tail.nsteps, minibatch order), the three-kernel step's
    statistics reductions, the step statistics and the state the call left.  keep_args: also the weights before the call
    and every argument.  tc_hook(orig, args): runs instead of the tensor-core launch."""
    from ddrl_b200 import kernels as K
    from ddrl_b200 import learner as LM
    GL = LM.GraphNetLearner
    orig = dict(learn=GL.learn_on_rollout, sgd=GL._sgd_phase, fwd=K.graphnet_forward, gae=K.gae, tc=K.graphnet_train_step_tc,
                red=LM._reduce_stats)
    cur = {}

    def learn(self, *args):
        rec = {"prep": True, "fwd": [], "launches": [], "reduce_calls": 0}
        cur["rec"] = rec
        if keep_args:
            rec["theta0"] = self.theta.detach().cpu().clone()
            rec["args"] = [a.detach().clone() for a in args]
        try:
            stats = orig["learn"](self, *args)
        finally:
            cur.clear()
        torch.cuda.synchronize()
        ss = self._tc["step_stats"] if self.step_kind == "tc" else rec.pop("ss_ref")
        rec.update(stats=stats, status=int(self.status.item()), sms=self.sms, ctas=self.ctas, step_kind=self.step_kind,
                   theta=self.theta[0].cpu().numpy().copy(), m=self.m[0].cpu().numpy().copy(),
                   v=self.v[0].cpu().numpy().copy(), beta_pow=self.beta_pow[0].cpu().numpy().copy(),
                   kl_coeff=self.kl_coeff.cpu().numpy().copy(), kl_coeff_host=float(self.kl_coeff_host[0]),
                   step_stats=ss.cpu().numpy().copy())
        log.append(rec)
        return stats

    def sgd(self, cols, perms, shuffle, R_):
        rec = cur["rec"]
        rec["prep"] = False
        rec["cols"] = {k: cols[k].detach().cpu().numpy().copy() for k in COLS}
        return orig["sgd"](self, cols, perms, shuffle, R_)

    def fwd(*a, **kw):
        out = orig["fwd"](*a, **kw)
        rec = cur.get("rec")
        if rec is not None and rec["prep"]:
            rec["fwd"].append(tuple(t.detach().cpu().numpy().copy() for t in out))
        return out

    def gae(*a, **kw):
        out = orig["gae"](*a, **kw)
        rec = cur.get("rec")
        if rec is not None:
            rec["gae"] = tuple(t.detach().cpu().numpy().copy() for t in out)      # before adv_standardize rescales adv
        return out

    def tc(*a, **kw):
        assert not kw
        rec = cur.get("rec")
        tail = a[20] if len(a) > 20 else None
        if rec is not None:
            rec["launches"].append(dict(R=int(a[2].shape[0]), A=int(a[10]), MB=int(a[11]), Gn=int(a[16]),
                                        nsteps=None if tail is None else int(tail.nsteps),
                                        mb_perm=None if a[12] is None else a[12].cpu().numpy().copy()))
        if tc_hook is not None:
            return tc_hook(orig["tc"], a)
        return orig["tc"](*a)

    def red(spart, step_stats, step_ctr):
        rec = cur.get("rec")
        if rec is not None:
            rec["reduce_calls"] += 1
            rec["ss_ref"] = step_stats
        return orig["red"](spart, step_stats, step_ctr)

    with pytest.MonkeyPatch.context() as mp:
        mp.setattr(GL, "learn_on_rollout", learn)
        mp.setattr(GL, "_sgd_phase", sgd)
        mp.setattr(K, "graphnet_forward", fwd)
        mp.setattr(K, "gae", gae)
        mp.setattr(K, "graphnet_train_step_tc", tc)
        mp.setattr(LM, "_reduce_stats", red)
        yield


def _assert_launch_shape(rec, E):
    """The launch shape this file claims to test; fails if the learner's choice or the kernel's row split drifts."""
    nb = rec["args"][9].shape[1] if "args" in rec else NB
    assert rec["sms"] == SMS, f"{rec['sms']} SMs: this file tests the 148-SM B200 launch shape"
    assert nb == NB and MB == 16384 and R == 524288
    if rec["step_kind"] != "tc":
        assert rec["launches"] == [] and rec["reduce_calls"] == E * NB, (rec["launches"], rec["reduce_calls"])
        assert rec["status"] == 0
        return
    assert len(rec["launches"]) == 1, "one persistent graphnet_train_step_tc launch per iteration"
    ln = rec["launches"][0]
    assert max(1, min(rec["ctas"], rec["sms"] // 2)) == ln["Gn"] == GN, (rec["ctas"], ln["Gn"])
    assert (ln["R"], ln["A"], ln["MB"], ln["nsteps"]) == (R, A, MB, E * NB), ln
    rows = _cta_rows(ln["MB"], ln["Gn"])
    assert _rpc(ln["MB"], ln["Gn"]) == 224
    assert [n for _, n in rows] == [224] * (GN - 1) + [32], rows
    assert rows[RAGGED_CTA] == (MB - 32, 32)
    assert rec["status"] == 0, f"tc status {rec['status']}"


def _run(inp, E, step="tc", iters=1, perms=None, tc_hook=None, bind=None):
    """A fresh GraphNetLearner (bench.py's arguments, step kind `step`) from the recorded weights, `iters` consecutive
    learn_on_rollout calls on the recorded rollout -> one record per call."""
    from ddrl_b200.config import PPOConfig
    from ddrl_b200.learner import GraphNetLearner
    L = GraphNetLearner(A, PPOConfig(num_sgd_iter=E, sgd_minibatch_size=R // NB), torch.device("cuda", 0),
                        theta=inp["theta0"], step=step)
    if bind is not None:
        bind(L)
    args = list(inp["args"])
    if perms is not None:
        args[9] = perms
    log = []
    with _instrumented(log, tc_hook=tc_hook):
        for _ in range(iters):
            L.learn_on_rollout(*args)
    for rec in log:
        _assert_launch_shape(rec, E)
    return log


# ---- bench.py's inputs ----------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def captured():
    """bench.time_graphnet(4096, E, steps=1, warmup=0) for E = 2 and 10, with learn_on_rollout recording its arguments
    (idx, state, adj, boot tensors, rewards, dones, eps, perms, shuffle), the weights before the call and what the call
    did and left -> {E: record}."""
    import bench
    torch.cuda.set_device(0)
    out = {}
    for E in (E_A, E_B):
        log = []
        with _instrumented(log, keep_args=True):
            bench.time_graphnet(ENVS, E, steps=1, warmup=0)
        assert len(log) == 1, len(log)
        out[E] = log[0]
    return out


def test_bench_launch_shape(captured):
    """bench.py's own calls: 148 SMs, Gn = 74 CTAs per net, MB = 16 384, nb = 32, the kernel's split 73 x 224 + 1 x 32 rows,
    ONE launch per iteration with tail.nsteps = E * nb, status 0; the two captures share the rollout."""
    for E, rec in captured.items():
        _assert_launch_shape(rec, E)
        assert rec["args"][9].shape == (E, NB)
        assert np.array_equal(rec["launches"][0]["mb_perm"], rec["args"][9].cpu().numpy().reshape(-1))
    a2, a10 = captured[E_A]["args"], captured[E_B]["args"]
    for i in range(9):                          # everything but perms and shuffle is drawn before them
        assert torch.equal(a2[i], a10[i]), i
    assert torch.equal(captured[E_A]["theta0"], captured[E_B]["theta0"])


# ---- the float64 oracle trajectory ---------------------------------------------------------------------------------------
def _host_inputs(rec):
    """A record's arguments on the host: the unshuffled [R] rows of the rollout, the [C] bootstrap rows and the rest."""
    idx, st, adj, bidx, bst, badj, rew, dones, eps, perms, shuffle = (a.cpu() for a in rec["args"])
    return dict(theta0=rec["theta0"].reshape(-1), idx=idx.reshape(R), st=st.reshape(R, 4, 23), adj=adj.reshape(R, 4, 4),
                bidx=bidx.reshape(C), bst=bst.reshape(C, 4, 23), badj=badj.reshape(C, 4, 4), rewards=rew.numpy(),
                dones=dones.numpy(), eps=eps.reshape(R, A), perms=perms.numpy(), shuffle=shuffle.long())


def _forward(theta, idx, st, adj, dt, chunk=CHUNK):
    """The oracle's GraphNet forward over many rows, `chunk` rows per call (the encoder's intermediate of 524 288 rows would
    take ~20 GB in float64)."""
    O = _oracle()
    lg, v = [], []
    with torch.no_grad():
        for r0 in range(0, st.shape[0], chunk):
            a, b = O.graphnet_forward(theta, idx[r0:r0 + chunk], st[r0:r0 + chunk].to(dt), adj[r0:r0 + chunk].to(dt), 2 * A)
            lg.append(a)
            v.append(b)
    return torch.cat(lg), torch.cat(v)


def _trajectory(h, dt, iters, E, mb=MB, chunk=CHUNK):
    """`iters` learner iterations on the same rollout in dtype dt, step by step, as GraphNetLearner.learn_on_rollout:
    forward + sample + bootstrap value, GAE (cols_per_env = 4), standardise, shuffle, E x nb steps (clip + TF1 Adam),
    KL-coefficient update.  -> one record per iteration; float64 adds the preparation phase, every step's statistics,
    the weights before the first and the last step, and `cut` = the first step with a row within NEAR_CLIP of the clip
    kink (`after_cut`: an earlier iteration had one)."""
    O = _oracle()
    cfg = O.PPOConfig(num_sgd_iter=E, sgd_minibatch_size=mb)
    f64 = dt == torch.float64
    n, ncol = h["st"].shape[0], h["bst"].shape[0]
    Tn = n // ncol
    theta, adam, klc = h["theta0"].to(dt), O.AdamState.zeros(h["theta0"].numel(), dt, cfg), cfg.kl_coeff
    sh = h["shuffle"]
    st_s, adj_s, idx_s = h["st"][sh].to(dt), h["adj"][sh].to(dt), h["idx"][sh]
    dones = np.repeat(h["dones"], ncol // h["dones"].shape[1], axis=1)
    out, forked = [], False
    for _ in range(iters):
        lg, v = _forward(theta, h["idx"], h["st"], h["adj"], dt, chunk)
        with torch.no_grad():
            act = O.dg_sample(lg, h["eps"].to(dt))
            logp = O.dg_logp(lg, act)
        _, vb = _forward(theta, h["bidx"], h["bst"], h["badj"], dt, chunk)
        adv, vt = O.gae_recurrence(h["rewards"], v.numpy().astype(np.float32).reshape(Tn, ncol), dones,
                                   vb.numpy().astype(np.float32), cfg.gamma, cfg.lambda_)
        adv_std = O.standardized(adv.reshape(-1).astype(np.float64) if f64 else adv.reshape(-1))
        b = {"actions": act, "old_logits": lg, "old_logp": logp, "vf_preds": v,
             "advantages": torch.from_numpy(np.asarray(adv_std)).to(dt), "value_targets": torch.from_numpy(vt.reshape(-1)).to(dt)}
        b = {k: x[sh] for k, x in b.items()}
        thetas, steps, cut, last = [], [], None, None
        for e in range(E):
            last = {k: [] for k in O.STAT_KEYS}
            for mbi in h["perms"][e]:
                rows = slice(int(mbi) * mb, (int(mbi) + 1) * mb)
                if f64:
                    thetas.append(theta)
                th = theta.clone().requires_grad_(True)
                lgm, vm = O.graphnet_forward(th, idx_s[rows], st_s[rows], adj_s[rows], 2 * A)
                loss, st = O.ppo_loss_from_outputs(lgm, vm, *(b[k][rows] for k in (
                    "actions", "old_logits", "old_logp", "vf_preds", "advantages", "value_targets")), klc, cfg)
                (g,) = torch.autograd.grad(loss, th)
                if f64 and cut is None:
                    near = _clip_branch(lgm.detach(), b["actions"][rows], b["old_logp"][rows], b["advantages"][rows], cfg)[2]
                    if bool(near.any()):
                        cut = len(steps)
                theta = O.adam_tf1_step(theta, O.clip_by_global_norm(g, cfg.grad_clip)[0], adam, cfg)
                st = {k: float(x.detach()) for k, x in st.items()}
                steps.append([st[k] for k in STEP_STATS])
                for k in O.STAT_KEYS:
                    last[k].append(st[k])
        stats = {k: float(np.mean(np.asarray(x, dtype=np.float32))) for k, x in last.items()}     # as O.sgd_loop
        klc = O.update_kl(klc, stats["kl"], cfg.kl_target)
        rec = dict(theta=theta.numpy().astype(np.float64), m=adam.m.numpy().astype(np.float64),
                   v=adam.v.numpy().astype(np.float64))
        if f64:
            a64 = adv.reshape(-1).astype(np.float64)
            rec.update(logits=lg.numpy(), value=v.numpy(), vboot=vb.numpy(), act=act.numpy(), logp=logp.numpy(),
                       gae_adv=adv.reshape(-1), vtarg=vt.reshape(-1), adv=np.asarray(adv_std),
                       moments=np.array([a64.size, a64.sum(), (a64 * a64).sum()]), step_stats=np.array(steps),
                       theta_first=thetas[0].numpy(), theta_last=thetas[-1].numpy(),
                       beta_pow=(adam.beta1_power, adam.beta2_power), kl_coeff=klc, stats=stats, cut=cut, after_cut=forked)
            forked = forked or cut is not None
        out.append(rec)
    return out


def _oracle_run(h, iters, E, mb=MB, chunk=CHUNK):
    """The float64 trajectory and its float32 twin side by side on two host threads -> one record per iteration (the
    twin's final state as twin_theta / twin_m / twin_v)."""
    threads = torch.get_num_threads()
    torch.set_num_threads(max(1, (os.cpu_count() or 1) // 2))
    try:
        with ThreadPoolExecutor(2) as ex:
            r64, r32 = ex.map(lambda dt: _trajectory(h, dt, iters, E, mb, chunk), (torch.float64, torch.float32))
    finally:
        torch.set_num_threads(threads)
    for a, b in zip(r64, r32):
        a.update(twin_theta=b["theta"], twin_m=b["m"], twin_v=b["v"])
    return r64


@pytest.fixture(scope="module")
def oracle(captured):
    """-> [iteration] records of the float64 trajectory of two iterations at E = 2 on bench's E = 2 rollout."""
    t0 = time.perf_counter()
    out = _oracle_run(_host_inputs(captured[E_A]), 2, E_A)
    print(f"\n[oracle] float64 trajectory + float32 twin, 2 iterations x {E_A * NB} steps of {MB} rows: "
          f"{time.perf_counter() - t0:.1f} s on {os.cpu_count()} host cores; clip-kink cut per iteration: "
          f"{[(r['cut'], r['after_cut']) for r in out]}")
    return out


# ---- A: trajectory -----------------------------------------------------------------------------------------------------------
def _device_step_stats(ss, mb=MB):
    """step_stats [steps, 1, 8] float64 sums over the minibatch rows -> [steps, 5] in STEP_STATS order."""
    s = np.asarray(ss, dtype=np.float64).reshape(-1, 8) / mb
    ev = np.maximum(-1.0, 1.0 - (s[:, 7] - s[:, 6] ** 2) / (s[:, 5] - s[:, 4] ** 2))
    return np.stack([s[:, 0], s[:, 1], s[:, 2], s[:, 3], ev], axis=-1)


def _update_err(theta, ref):
    """max |theta - theta64| over the size of the float64 update of the iteration."""
    upd = ref["theta"] - ref["theta_first"]
    return float(np.abs(np.asarray(theta, dtype=np.float64) - ref["theta"]).max() / np.abs(upd).max())


def _prep_errors(rec, ref):
    """The preparation phase of one learn_on_rollout call, unshuffled, against the float64 record -> {name: error}."""
    cols = rec["cols"]
    (lg, v), (_, vb) = rec["fwd"][0], rec["fwd"][1]
    gadv, gvt, mom = rec["gae"]
    dev = dict(logits=lg, value=v, vboot=vb, act=cols["act"], logp=cols["logp"], vtarg=cols["vtarg"], adv=cols["adv"],
               gae_adv=gadv.reshape(-1))
    err = {k: scaled_err(x.reshape(ref[k].shape), ref[k]) for k, x in dev.items()}
    assert np.array_equal(gvt.reshape(-1), cols["vtarg"]) and np.array_equal(cols["value"], v)
    m, m64 = np.asarray(mom, dtype=np.float64).reshape(3), ref["moments"]
    std64 = np.sqrt(m64[2] / m64[0] - (m64[1] / m64[0]) ** 2)
    err["moments"] = max(abs(m[1] - m64[1]) / m64[0] / std64, abs(m[2] - m64[2]) / m64[2]) if m[0] == m64[0] else np.inf
    return err


def _compare(rec, ref, it, tag):
    """One learn_on_rollout record against the oracle's iteration `it` -> (failures, first off step or None, measurements).
    Prints one line with the measured errors.  If the reference trajectory reached a row at the clip kink, the step
    statistics are compared up to that step and nothing that depends on the update; the beta powers and the status are
    checked always."""
    fails = []

    def check(ok, msg):
        if not ok:
            fails.append(f"{tag} it {it}: {msg}")
    ss = _device_step_stats(rec["step_stats"])
    ratio = _stat_ratio(ss, ref["step_stats"], STAT_TOL_A)
    if ref["after_cut"]:
        ratio[:] = 0.0
    elif ref["cut"] is not None:
        ratio[ref["cut"] + 1:] = 0.0
    bad = np.flatnonzero(ratio > 1.0)
    first = int(bad[0]) if len(bad) else None
    if first is not None:
        fails.append(f"{tag} it {it}: step statistics first off at step {first} (error / tolerance {ratio[first]:.3g})")
    steps = len(ratio)
    beta = _beta_chain(steps * (it + 1))
    check(rec["beta_pow"][0] == beta[0] and rec["beta_pow"][1] == beta[1], f"beta powers {rec['beta_pow']} != {beta}")
    check(rec["status"] == 0, f"status {rec['status']}")
    meas = dict(stat=float(ratio.max()), cut=ref["cut"], after_cut=ref["after_cut"])
    if ref["after_cut"]:
        print(f"[A {tag} it={it}] weight-dependent checks skipped: an earlier iteration reached the clip kink")
        return fails, first, meas
    prep = _prep_errors(rec, ref)
    for k, e in prep.items():
        check(e < PREP_TOL[k], f"{k} error {e:.3g} >= {PREP_TOL[k]}")
    meas["prep"] = prep
    ptxt = " ".join(f"{k}={e:.3g}" for k, e in prep.items())
    if ref["cut"] is not None:
        print(f"[A {tag} it={it}] prep: {ptxt}; step statistics compared up to step {ref['cut']} (a row at the clip kink), "
              f"step_stats_err/tol={meas['stat']:.3g}")
        return fails, first, meas
    upd, twin = _update_err(rec["theta"], ref), _update_err(ref["twin_theta"], ref)
    bound = max(10.0 * twin, UPD_FLOOR)
    guard = _update_err(ref["theta_last"], ref)          # the float64 trajectory without its last step
    check(guard > 10.0 * bound, f"last-step guard {guard:.3g} is not 10x above the bound {bound:.3g}")
    check(upd < bound, f"update error {upd:.3g} >= {bound:.3g} (twin {twin:.3g})")
    em, ev_ = scaled_err(rec["m"], ref["m"]), scaled_err(rec["v"], ref["v"])
    em_t, ev_t = scaled_err(ref["twin_m"], ref["m"]), scaled_err(ref["twin_v"], ref["v"])
    check(em < max(10.0 * em_t, MV_FLOOR), f"adam m error {em:.3g} (twin {em_t:.3g})")
    check(ev_ < max(10.0 * ev_t, MV_FLOOR), f"adam v error {ev_:.3g} (twin {ev_t:.3g})")
    check(rec["kl_coeff_host"] == ref["kl_coeff"] and rec["kl_coeff"][0] == np.float32(ref["kl_coeff"]),
          f"kl coefficient {rec['kl_coeff_host']} / {rec['kl_coeff'][0]} != {ref['kl_coeff']}")
    stat_err = 0.0
    for k, rv in ref["stats"].items():
        e = abs(rec["stats"][0][k] - rv) / max(1.0, abs(rv))
        stat_err = max(stat_err, e)
        check(e < 1e-4, f"returned {k} {rec['stats'][0][k]} != {rv}")
    meas.update(upd=upd, twin=twin, bound=bound, guard=guard, m=em, v=ev_, m_twin=em_t, v_twin=ev_t, ret=stat_err)
    print(f"[A {tag} it={it}] prep: {ptxt}; update_err={upd:.3g} twin={twin:.3g} bound={bound:.3g} guard={guard:.3g} "
          f"step_stats_err/tol={meas['stat']:.3g} m_err={em:.3g} (twin {em_t:.3g}) v_err={ev_:.3g} (twin {ev_t:.3g}) "
          f"returned_stats_err={stat_err:.3g} (tol 1e-4) kl_coeff={rec['kl_coeff_host']}")
    return fails, first, meas


@pytest.mark.parametrize("step", ["tc", "three-kernel"])
def test_two_iterations_match_oracle(step, captured, oracle):
    """Two consecutive E = 2 iterations on bench's rollout, as bench.py's timed loop runs them: preparation phase, the
    64 steps' loss statistics and the final weights / Adam state / beta powers / KL coefficient / returned stats of each,
    against the float64 trajectory."""
    log = _run(captured[E_A], E_A, step, iters=2)
    fails = []
    for it, rec in enumerate(log):
        fails += _compare(rec, oracle[it], it, step)[0]
    assert not fails, "\n".join(fails)


def test_one_repeated_minibatch_is_caught(captured, oracle):
    """Negative control: step 40 (epoch 1, position 8) repeats the minibatch of step 39.  A must flag step 40 first (the
    steps before it pass) and the final weights of the iteration."""
    ref = oracle[0]
    target = 40
    assert ref["cut"] is None or ref["cut"] > target, f"the reference reaches the clip kink at step {ref['cut']}"
    perms = captured[E_A]["args"][9].clone()
    e, i = divmod(target, NB)
    assert perms[e, i] != perms[e, i - 1]
    perms[e, i] = perms[e, i - 1]
    (rec,) = _run(captured[E_A], E_A, "tc", perms=perms)
    fails, first, meas = _compare(rec, ref, 0, "fault")
    assert first == target, (first, fails)
    if ref["cut"] is None:
        assert meas["upd"] > 10.0 * meas["bound"], meas


# ---- B: teacher-forced steps at E = 10 ---------------------------------------------------------------------------------------
def _snap(L):
    torch.cuda.synchronize()
    return {k: getattr(L, k).cpu().numpy().astype(np.float64).copy()
            for k in ("theta", "m", "v", "beta_pow", "kl_coeff", "grad", "gnorm")}


@pytest.fixture(scope="module")
def teacher_forced(captured):
    """The E = 10 iteration on bench's rollout, its one persistent launch run as 320 single-step launches of
    graphnet_train_step_tc (tail.nsteps = 1) on the learner's own buffers; mb_perm / step_ctr advance as in the persistent
    launch.  Snapshots of the state around the SAMPLED steps, the shuffled columns the learner passed in, and at
    CONTROL_STEP three extra launches from a copy of the pre-step state: unmodified, with adv zeroed on the rows of the
    ragged CTA, with adv x 2^8 on the second tile of CTA STRESS_CTA."""
    from ddrl_b200 import kernels as K
    out = {"pre": {}, "post": {}, "copy": {}}
    box = {}

    def bind(L):
        box["L"] = L

    def hook(orig, a):
        L = box["L"]
        a = list(a)
        tail = a[20]
        n = int(tail.nsteps)
        assert n == E_B * NB
        out["cols"] = {k: t.cpu() for k, t in zip(("idx", "st", "adj") + COLS, a[1:10])}
        out["mb_perm"] = a[12].cpu().numpy().copy()
        cfg = L.cfg
        for s in range(n):
            tail.nsteps = 1
            if s in SAMPLED:
                out["pre"][s] = _snap(L)
            if s == CONTROL_STEP:
                mb = int(out["mb_perm"][s])
                r0 = mb * MB
                zero = a[8].clone()
                rows = _cta_rows(MB, GN)[RAGGED_CTA]
                zero[r0 + rows[0]:r0 + rows[0] + rows[1]] = 0.0
                big = a[8].clone()
                c0 = _cta_rows(MB, GN)[STRESS_CTA][0]
                big[r0 + c0 + 64:r0 + c0 + 128] *= 256.0
                out["stress_rows"] = (c0 + 64, c0 + 128)
                for name, adv in (("same", a[8]), ("ragged_lost", zero), ("stress", big)):
                    th, m, v, bp = (t.clone() for t in (L.theta, L.m, L.v, L.beta_pow))
                    grad, gn = torch.zeros_like(L.grad), torch.zeros_like(L.gnorm)
                    w = L._tc
                    bar, sq = torch.zeros_like(w["tail_bar"]), torch.zeros_like(w["tail_sq"])
                    ctr = torch.full((1,), s, dtype=torch.int32, device=L.device)
                    status = torch.zeros(1, dtype=torch.int32, device=L.device)
                    ss = torch.zeros_like(w["step_stats"])
                    tl = K.make_sgd_tail(th, m, v, bp, grad, bar, sq, cfg.lr, cfg.beta1, cfg.beta2, cfg.adam_eps, cfg.grad_clip,
                                         gn, step_stats=ss, step_ctr=ctr, status=status)
                    b = list(a)
                    b[0], b[8], b[13] = th.reshape(-1), adv, ctr
                    b[17], b[18], b[19], b[20] = torch.empty_like(w["grad_part"]), torch.zeros_like(w["stat_part"]), status, tl
                    orig(*b)
                    torch.cuda.synchronize()
                    out["copy"][name] = dict(grad=grad[0].cpu().numpy().astype(np.float64), status=int(status.item()),
                                             step_stats=ss[s].cpu().numpy().copy(), adv=adv.cpu() if name != "same" else None)
            orig(*a)
            if s in SAMPLED:
                out["post"][s] = _snap(L)
        tail.nsteps = n

    (rec,) = _run(captured[E_B], E_B, "tc", tc_hook=hook, bind=bind)
    out["rec"] = rec
    return out


def _gn_loss_grad(theta, cols, rows, klc, cfg, dtype, adv=None):
    """autograd of the mean PPO loss over cols[*][rows] at theta -> (reference gradients, [5] stats in STEP_STATS order,
    max |v|).  The first gradient is torch's; float64 adds one per non-empty subset of the rows within NEAR_CLIP of the
    clip kink, with those rows on the other side of it (as test_gpu_bench_workload._loss_grad)."""
    O = _oracle()
    th = torch.from_numpy(np.asarray(theta)).to(dtype).requires_grad_(True)
    c = {k: cols[k][rows].to(dtype) for k in ("st", "adj") + COLS}
    if adv is not None:
        c["adv"] = adv[rows].to(dtype)
    lg, v = O.graphnet_forward(th, cols["idx"][rows], c["st"], c["adj"], 2 * A)
    loss, st = O.ppo_loss_from_outputs(lg, v, c["act"], c["logits"], c["logp"], c["value"], c["adv"], c["vtarg"], klc, cfg)
    near_rows = []
    if dtype == torch.float64:
        ratio, flows, near = _clip_branch(lg, c["act"], c["logp"], c["adv"], cfg)
        near_rows = near.nonzero().reshape(-1).tolist()
        assert len(near_rows) <= 3, f"{len(near_rows)} rows at the clip kink"
    (g,) = torch.autograd.grad(loss, th, retain_graph=bool(near_rows))
    deltas = []
    for i, r in enumerate(near_rows):
        (d,) = torch.autograd.grad(c["adv"][r] * ratio[r], th, retain_graph=i + 1 < len(near_rows))
        deltas.append((d if bool(flows[r]) else -d) / ratio.numel())
    refs = [g + sum(sub, torch.zeros_like(g)) for k in range(len(deltas) + 1) for sub in itertools.combinations(deltas, k)]
    return ([x.detach().numpy().astype(np.float64) for x in refs], np.array([float(st[k].detach()) for k in STEP_STATS]),
            float(v.detach().abs().max()))


def _shapes():
    O = _oracle()
    return [shp for _, shp in O.graphnet_shapes(2 * A)] + [shp for _, shp in O.graphnet_shapes(1)]


def _grad_check(grad, refs, g32_refs, vmax, cfg):
    """B's gradient rule -> (scaled error, value-bias error over its allowance, AssertionError or None).  Rows at the
    clip kink: the side the kernel took, and the twin's round-off around the side it took.  The critic's linear_out/bias
    gradient is vf_loss_coeff * 2 * mean(v - R): its error is the mean error of the value forward, so it may be off by
    2 * vf_loss_coeff * FWD_TOL * max|v|."""
    g64 = min(refs, key=lambda x: scaled_err(grad, x))
    twin = g32_refs[0] - min(refs, key=lambda x: scaled_err(g32_refs[0], x)) + g64
    vb_off = grad.size - 1
    vb_allow = 2.0 * cfg.vf_loss_coeff * FWD_TOL * vmax
    try:
        assert_grad_per_variable(grad, g64, twin, _shapes(), TC_GRAD_TOL, allow={vb_off: vb_allow})
        exc = None
    except AssertionError as e:
        exc = e
    return scaled_err(grad, g64), abs(grad[vb_off] - g64[vb_off]) / vb_allow, exc


def _references(tf, steps, extra=()):
    """float64 and float32 autograd at the device's weights before each step of `steps` (+ `extra`: (name, step, adv)),
    on the device's shuffled columns, on host threads -> {key: (refs64, stats64, vmax, refs32)}."""
    cfg = _cfg_o(E_B)
    cols = tf["cols"]
    memo = tf.setdefault("refs", {})
    jobs = [j for j in [(s, s, None) for s in steps] + list(extra) if j[0] not in memo]

    def one(job):
        key, s, adv = job
        pre = tf["pre"][s]
        mb = int(tf["mb_perm"][s])
        rows = slice(mb * MB, (mb + 1) * MB)
        th, klc = pre["theta"][0], float(pre["kl_coeff"][0])
        refs, st64, vmax = _gn_loss_grad(th, cols, rows, klc, cfg, torch.float64, adv)
        r32, _, _ = _gn_loss_grad(th, cols, rows, klc, cfg, torch.float32, adv)
        return key, (refs, st64, vmax, r32)
    workers = 3
    threads = torch.get_num_threads()
    torch.set_num_threads(max(1, (os.cpu_count() or 1) // workers))
    try:
        with ThreadPoolExecutor(workers) as ex:
            memo.update(ex.map(one, jobs))
    finally:
        torch.set_num_threads(threads)
    return {j[0]: memo[j[0]] for j in [(s, s, None) for s in steps] + list(extra)}


def test_sampled_steps_match_oracle_at_device_weights(teacher_forced):
    """B: at steps 0, 1, 31, 32, 63, 64, 159, 288, 319 of the E = 10 iteration (single-step launches, teacher-forced): the
    reduced gradient per variable against float64 autograd at the device's weights on the device's own shuffled columns,
    the device's clip + TF1 Adam against float64 arithmetic from its own gradient and state, and the step's statistics."""
    tf = teacher_forced
    cfg = _cfg_o(E_B)
    f32 = lambda x: float(np.float32(x))
    b1, b2, lr, eps, clip = (f32(x) for x in (cfg.beta1, cfg.beta2, cfg.lr, cfg.adam_eps, cfg.grad_clip))
    ss_all = _device_step_stats(tf["rec"]["step_stats"])
    refs = _references(tf, SAMPLED)
    fails = []
    for s in SAMPLED:
        pre, post = tf["pre"][s], tf["post"][s]
        r64, st64, vmax, r32 = refs[s]
        grad = post["grad"][0]
        e, vb, exc = _grad_check(grad, r64, r32, vmax, cfg)
        if e >= TC_GRAD_TOL:
            fails.append(f"step {s}: gradient error {e:.3g} >= {TC_GRAD_TOL}")
        if exc is not None:
            fails.append(f"step {s}: gradient per variable: {exc}")
        # global-norm clip + TF1 Adam in float64 from the device's own gradient and state
        th0, m0, v0, bp0 = pre["theta"][0], pre["m"][0], pre["v"][0], pre["beta_pow"][0]
        norm = float(np.sqrt((grad ** 2).sum()))
        gc = grad * (clip * min(1.0 / norm, 1.0 / clip))
        lr_t = lr * np.sqrt(1.0 - bp0[1]) / (1.0 - bp0[0])
        m = m0 + (gc - m0) * (1.0 - b1)
        v = v0 + (gc * gc - v0) * (1.0 - b2)
        th = th0 - (m * lr_t) / (np.sqrt(v) + eps)
        errs = dict(gnorm=abs(post["gnorm"][0] - norm) / norm, m=scaled_err(post["m"][0], m), v=scaled_err(post["v"][0], v),
                    theta=float((np.abs(post["theta"][0] - th) / (5e-7 * np.abs(th) + 1e-9)).max()))    # rtol 5e-7, atol 1e-9
        for k, x in errs.items():
            if x >= (1.0 if k == "theta" else 1e-6):
                fails.append(f"step {s}: tail arithmetic: {k} error {x:.3g}")
        bp1 = post["beta_pow"][0]
        if not (bp1[0] == np.float32(np.float32(bp0[0]) * np.float32(b1)) and bp1[1] == np.float32(np.float32(bp0[1]) * np.float32(b2))):
            fails.append(f"step {s}: beta powers {bp0} -> {bp1}")
        x = float(_stat_ratio(ss_all[s], st64, STAT_TOL_B))
        if x > 1.0:
            fails.append(f"step {s}: step statistics error / tolerance {x:.3g}: {ss_all[s]} vs {st64}")
        print(f"[B s={s}] minibatch={int(tf['mb_perm'][s])} grad_err={e:.3g} (tol {TC_GRAD_TOL}) "
              f"value_bias_err/allow={vb:.3g} gnorm_err={errs['gnorm']:.3g} m_err={errs['m']:.3g} v_err={errs['v']:.3g} "
              f"theta_err/tol={errs['theta']:.3g} step_stats_err/tol={x:.3g} rows_at_the_clip_kink={len(r64).bit_length() - 1}")
    assert tf["rec"]["status"] == 0
    assert not fails, "\n".join(fails)


# ---- C: bit-identity ---------------------------------------------------------------------------------------------------------
_STATE = ("theta", "m", "v", "beta_pow", "kl_coeff", "step_stats")


def test_persistent_launch_equals_single_step_launches(captured, teacher_forced):
    """The one persistent 320-step launch bench.py timed leaves the same bits as B's 320 single-step launches: weights,
    Adam moments, beta powers, every step's statistics and the KL coefficient."""
    a, b = captured[E_B], teacher_forced["rec"]
    for k in _STATE:
        assert np.array_equal(a[k], b[k]), k
    assert a["stats"] == b["stats"] and a["kl_coeff_host"] == b["kl_coeff_host"]


def test_repeated_iteration_is_bit_identical(captured):
    """The same E = 10 iteration from the same state gives identical bits (the tail's reductions have a fixed order)."""
    (b,) = _run(captured[E_B], E_B, "tc")
    a = captured[E_B]
    for k in _STATE:
        assert np.array_equal(a[k], b[k]), k
    assert a["stats"] == b["stats"]


# ---- D: controls of B, and the first-tile gradient scale ---------------------------------------------------------------------
def test_copied_launch_reproduces_the_step(teacher_forced):
    """The harness of the controls: the launch at CONTROL_STEP repeated from a copy of the pre-step state gives the step's
    own gradient and statistics bit for bit."""
    tf = teacher_forced
    same = tf["copy"]["same"]
    assert same["status"] == 0
    assert np.array_equal(same["grad"], tf["post"][CONTROL_STEP]["grad"][0])
    assert np.array_equal(same["step_stats"], tf["rec"]["step_stats"][CONTROL_STEP])


def test_lost_ragged_cta_is_caught(teacher_forced):
    """Negative control: the launch of CONTROL_STEP with adv zeroed on the 32 rows of CTA 73 (one ragged CTA of 148) is
    compared with the unmodified float64 reference; B's gradient check must fail."""
    tf = teacher_forced
    cfg = _cfg_o(E_B)
    (ref,) = _references(tf, (CONTROL_STEP,)).values()
    r64, _, vmax, r32 = ref
    c = tf["copy"]["ragged_lost"]
    e, vb, exc = _grad_check(c["grad"], r64, r32, vmax, cfg)
    print(f"[D ragged CTA {RAGGED_CTA} lost, step {CONTROL_STEP}] grad_err={e:.3g} (tol {TC_GRAD_TOL}) status={c['status']} "
          f"check: {'FAILED as required: ' + str(exc) if exc is not None else 'passed'}")
    assert exc is not None, "B's check does not see the 32 rows of the ragged CTA"


def test_second_tile_gradient_scale_stress(teacher_forced):
    """Stress of the per-CTA gradient scale taken from the first tile only: the launch of CONTROL_STEP with adv x 2^8 on
    the second tile of CTA 0 against a float64 reference built on the same scaled inputs.  Either the kernel flags the
    fp16 range (status bit 8, dl overflow) or the gradient passes B's check: a wrong gradient with status 0 is a bug."""
    tf = teacher_forced
    cfg = _cfg_o(E_B)
    c = tf["copy"]["stress"]
    (ref,) = _references(tf, (), extra=[("stress", CONTROL_STEP, c["adv"])]).values()
    r64, _, vmax, r32 = ref
    e, vb, exc = _grad_check(c["grad"], r64, r32, vmax, cfg)
    print(f"[D stress: adv x 256 on rows {tf['stress_rows']} of the minibatch (tile 2 of CTA {STRESS_CTA}), step "
          f"{CONTROL_STEP}] status={c['status']} grad_err={e:.3g} (tol {TC_GRAD_TOL}) check: "
          f"{'passed' if exc is None else 'failed: ' + str(exc)}")
    assert (c["status"] & 8) or exc is None, f"status {c['status']} and a wrong gradient: {exc}"

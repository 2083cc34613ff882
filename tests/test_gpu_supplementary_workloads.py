"""The other FCNet configurations bench.py times (`run_supplementary`) against the float64 oracle, at their own shapes and
with bench.py's own inputs for them.

bench.time_fcnet(arch, envs, nb, "tc", ...) trains with FCNetLearner's defaults: the tensor-core step and the atomic
partial-gradient reduction.  On a 148-SM B200 the four configurations run these launch shapes:

- C1, the reference's own minibatch shape (RLlib's sgd_minibatch_size = 128), FullyDecentral (P 4, D 19, A 2) and
  Centralized (P 1, D 43, A 8): 500 envs x T = 32 = 16 000 rows per policy, 125 minibatches of 128 rows, G = 32 CTAs per
  policy with rpc = 8 rows each: CTAs 0..15 hold one ragged 8-row tile, CTAs 16..31 no rows (they still own a slice of
  the fused tail), and all 1 250 steps of an iteration run in ONE persistent launch.  TF1 Adam's beta1 power enters the
  float32 subnormal range at step 829 and stays at its fixed point 4 * 2^-149 from step 965, inside the first launch.
- Local (P 4, D 35, A 2) and Centralized (P 1, D 43, A 8) at bench's 4096 envs: 131 072 rows per policy, 32 minibatches
  of 4096 rows, G = 32 CTAs with one full 128-row tile each, 320 steps in one launch.  Both are the ping-pong kernel's
  KX = 48 layouts; Centralized (A = 8) is its tightest one: the staged old logits move into the W1 region and the
  head-bias sums stay in shared memory.

Each configuration gets the headline's checks (tests/test_gpu_bench_workload.py), in the tc-atomic, tc-fixed and fp32
modes:
- A: three iterations on rollout sets 0, 1, 0 (time_fcnet's untimed calls: eager, capture of set 1, capture of set 0)
  against the float64 trajectory: filter, preparation phase, every step's loss statistics, and after each iteration the
  weights, Adam state, bit-exact beta powers, KL coefficient and returned statistics.
- B: every step of the first iteration teacher-forced at the device's weights: gradient per variable, clip + TF1 Adam,
  beta powers, step statistics.
- C: with the fixed-order reduction the persistent launch is bit-identical to one launch per step.
- D: a repeated minibatch in one policy must be flagged by A at its step and policy, and a step with the advantages
  zeroed on the rows of the last CTA that holds rows must fail B's gradient check.

Measured errors of these checks on a B200: profiles/r09_supplementary_workload_errors.txt."""
import contextlib

import numpy as np
import pytest
import torch

from tests.test_gpu_bench_workload import (MODES, SMS, Workload, _assert_bench_shape, _cfg_o, _learn, _learner,
                                           _step_rows, _to_dev, check_every_step, check_iterations,
                                           check_persistent_equals_one_step, check_repeated_minibatch, compared_steps,
                                           cta_rows, grad_check, oracle_trajectory)

pytestmark = pytest.mark.gpu

# bench.run_supplementary's FCNet jobs that this file covers: name -> time_fcnet's (arch, envs, minibatches per epoch, mode)
JOBS = {"C1_reference_minibatch_shape_FullyDecentral_16000rows_MB128": ("FullyDecentral", 500, 125, "tc"),
        "C1_Centralized_16000rows_MB128": ("Centralized", 500, 125, "tc"),
        "C3_Local": ("Local", 4096, 32, "tc"),
        "Centralized": ("Centralized", 4096, 32, "tc")}
# the jobs of run_supplementary covered elsewhere: name -> (test module, test, parameter)
COVERED_ELSEWHERE = {"FullyDecentral_fp32_parity_kernel": ("tests.test_gpu_bench_workload",
                                                           "test_bench_workload_iterations_match_oracle", "fp32"),
                     "C4_shared_GraphNet": ("tests.test_gpu_graphnet_workload", "test_two_iterations_match_oracle", None)}
IDS = {"C1_reference_minibatch_shape_FullyDecentral_16000rows_MB128": "C1_FullyDecentral",
       "C1_Centralized_16000rows_MB128": "C1_Centralized", "C3_Local": "Local", "Centralized": "Centralized"}
JOB_OF = {v: k for k, v in IDS.items()}
# per job: what _sgd_setup returns (MB, nb, G) for the tensor-core and the fp32 step on a 148-SM B200, the rows of each
# tensor-core CTA, (policy, step) of the repeated-minibatch control (a step before the policy's first row at the clip
# kink, at a position > 0 of its epoch) and the step of the lost-CTA control
C1_ROWS = (8,) * 16 + (0,) * 16
EXPECT = {
    "C1_reference_minibatch_shape_FullyDecentral_16000rows_MB128":
        dict(tc_setup=(128, 125, 32), tc_rows=C1_ROWS, fp32_setup=(128, 125, 8), control=(2, 700), lost_cta_step=1000),
    "C1_Centralized_16000rows_MB128":
        dict(tc_setup=(128, 125, 32), tc_rows=C1_ROWS, fp32_setup=(128, 125, 8), control=(0, 700), lost_cta_step=1000),
    "C3_Local":
        dict(tc_setup=(4096, 32, 32), tc_rows=(128,) * 32, fp32_setup=(4096, 32, 37), control=(2, 200), lost_cta_step=200),
    "Centralized":
        dict(tc_setup=(4096, 32, 32), tc_rows=(128,) * 32, fp32_setup=(4096, 32, 148), control=(0, 150), lost_cta_step=200),
}
ITER_SETS = (0, 1, 0)      # time_fcnet's untimed calls with its two rollout sets


# ---- bench.py's inputs ----------------------------------------------------------------------------------------------------
@contextlib.contextmanager
def _recording(log):
    """Wraps FCNetLearner.learn_on_rollout: every call appends the weights before it, the learner's PPOConfig and shapes,
    the launch shape it chose and a host copy of its arguments."""
    from ddrl_b200.learner import FCNetLearner
    orig = FCNetLearner.learn_on_rollout

    def learn(self, *args, **kw):
        assert not kw and len(args) == 7, "time_fcnet passes the seven rollout tensors"
        R = args[0].shape[1] * args[0].shape[2]
        MB, nb, G = self._sgd_setup(R)
        log.append(dict(theta0=self.theta.detach().cpu().clone(), cfg=self.cfg, P=self.P, D=self.D, A=self.A, mode=self.mode,
                        setup=(MB, nb, G), persistent=self._persistent_steps(G), atomic=self.atomic_reduce,
                        fuse_tail=self.fuse_tail, sms=self.sms,
                        args=dict(zip(("raw", "boot", "rewards", "dones", "eps", "perms", "shuffle"),
                                      (a.detach().cpu().clone() for a in args)))))
        return orig(self, *args)

    with pytest.MonkeyPatch.context() as mp:
        mp.setattr(FCNetLearner, "learn_on_rollout", learn)
        yield


@pytest.fixture(scope="module")
def captured():
    """bench.time_fcnet(arch, envs, nb, mode, steps=1, warmup=0) of every job, recorded -> {job: [one record per
    learn_on_rollout call]}: three untimed calls on rollout sets 0, 1, 0, then the timed one."""
    import bench
    torch.cuda.set_device(0)
    out = {}
    for name, (arch, envs, nb, mode) in JOBS.items():
        log = []
        with _recording(log):
            bench.time_fcnet(arch, envs, nb, mode, steps=1, warmup=0)
        assert len(log) == 4, len(log)
        out[name] = log
        torch.cuda.empty_cache()
    return out


def test_bench_launch_shape(captured):
    """What bench.py's own learner chose for every job: the tensor-core step with the atomic reduction, the fused tail,
    the expected (MB, nb, G) and row split on 148 SMs, one persistent launch per iteration; time_fcnet's untimed calls
    visit rollout sets 0, 1, 0 and the first starts from the initial weights."""
    for name, log in captured.items():
        ex = EXPECT[name]
        rec = log[0]
        assert rec["sms"] == SMS, rec["sms"]
        assert rec["mode"] == "tc" and rec["atomic"] and rec["fuse_tail"], name
        assert rec["setup"] == ex["tc_setup"] and cta_rows(*rec["setup"][::2]) == ex["tc_rows"], (name, rec["setup"])
        assert rec["persistent"] and ex["tc_setup"][2] * rec["P"] <= SMS, name
        for k in rec["args"]:
            assert torch.equal(log[2]["args"][k], rec["args"][k]), (name, k)
        assert not torch.equal(log[1]["args"]["raw"], rec["args"]["raw"]), name
        assert not torch.equal(log[1]["theta0"], rec["theta0"]), name


def _workload(name, log):
    """The Workload record of a job from bench's recorded calls."""
    from ddrl_b200.config import PPOConfig
    rec = log[0]
    P, T, C, D = rec["args"]["raw"].shape
    E, NB = rec["args"]["perms"].shape[1:]
    A = rec["args"]["eps"].shape[-1]
    MB = rec["cfg"].sgd_minibatch_size
    assert (P, D, A) == (rec["P"], rec["D"], rec["A"]) and MB * NB == T * C
    assert rec["cfg"] == PPOConfig(num_sgd_iter=E, sgd_minibatch_size=MB), rec["cfg"]     # the oracle's hyper-parameters
    return Workload(name=IDS[name], P=P, D=D, A=A, T=T, C=C, E=E, NB=NB, MB=MB, sets=[log[0]["args"], log[1]["args"]],
                    iter_sets=ITER_SETS, theta0=rec["theta0"], tc_setup=EXPECT[name]["tc_setup"],
                    tc_rows=EXPECT[name]["tc_rows"], fp32_setup=EXPECT[name]["fp32_setup"], control=EXPECT[name]["control"])


@pytest.fixture(scope="module", params=list(JOBS), ids=list(IDS.values()))
def workload(request, captured):
    return _workload(request.param, captured[request.param])


@pytest.fixture(scope="module")
def oracle(workload):
    """-> [iteration][policy] records of the workload's float64 trajectory (+ the float32 twin's end state)."""
    return oracle_trajectory(workload)


# ---- A, B, C: the headline's checks at each configuration -------------------------------------------------------------------
@pytest.mark.parametrize("mode", list(MODES))
def test_iterations_match_oracle(mode, workload, oracle):
    """A: three bench-shaped iterations (sets 0, 1, 0) against the float64 trajectory; prints how many steps of each
    policy and iteration were compared (a row at the clip kink ends a policy's comparison)."""
    w = workload
    fails = check_iterations(w, mode, oracle, f"{w.name} {mode}")
    for it, refs in enumerate(oracle):
        print(f"[A {w.name} {mode} it={it}] steps compared per policy (of {w.STEPS}): "
              f"{[compared_steps(w, r) for r in refs]}")
    assert not fails, "\n".join(fails)


@pytest.mark.parametrize("mode", list(MODES))
def test_every_step_matches_oracle_at_device_weights(mode, workload):
    """B: every step of the first iteration (1 250 at C1, 320 otherwise), one eager launch per step, teacher-forced at
    the device's weights."""
    w = workload
    fails = check_every_step(w, mode, f"{w.name} {mode}")
    assert not fails, "\n".join(fails)


def test_persistent_launch_equals_one_step_launches(workload):
    """C: fixed-order reduction, the persistent launch of all steps of an iteration against one eager launch per step:
    bit-identical state after each of the three iterations."""
    check_persistent_equals_one_step(workload)


# ---- D: negative controls -----------------------------------------------------------------------------------------------
def test_one_repeated_minibatch_is_caught(workload, oracle):
    """D1: in the first iteration, one policy's step repeats the minibatch of its previous step; A must flag exactly that
    step and policy, and pass the other policies."""
    w = workload
    check_repeated_minibatch(w, oracle, f"{w.name} fault")


@pytest.mark.parametrize("mode", [m for m in MODES if MODES[m]["mode"] == "tc"])
def test_lost_cta_is_caught(mode, workload):
    """D2: one teacher-forced step of the first iteration runs with the advantages zeroed on the rows of the last CTA
    that holds rows (CTA 15's 8 rows at C1, CTA 31's 128 rows otherwise), in every policy; against the unmodified float64
    reference B's gradient check must fail for every policy."""
    w = workload
    cfg = _cfg_o(w)
    last = max(i for i, n in enumerate(w.tc_rows) if n)
    r0, n = sum(w.tc_rows[:last]), w.tc_rows[last]
    target = EXPECT[JOB_OF[w.name]]["lost_cta_step"]
    r = w.sets[w.iter_sets[0]]
    perms = r["perms"].numpy()
    L = _learner(w, mode, persistent=False, use_graph=False)
    _assert_bench_shape(w, L, mode, persistent=False)
    orig = L._sgd_step
    ctx = {"step": 0}

    def step(b, MB_, G, hyper, src, nsteps=1):
        s = ctx["step"]
        ctx["step"] += 1
        if s != target:
            return orig(b, MB_, G, hyper, src, nsteps)
        torch.cuda.synchronize()
        ctx["pre"] = (L.theta.cpu().numpy().astype(np.float64), L.kl_coeff.cpu().numpy().astype(np.float64))
        ctx["cols"] = {k: src[k].cpu() for k in ("obs", "act", "logits", "logp", "value", "adv", "vtarg")}
        adv = src["adv"]
        keep = adv.clone()
        for p in range(w.P):
            rows = _step_rows(w, perms, p, s)
            adv[p, rows.start + r0:rows.start + r0 + n] = 0.0
        orig(b, MB_, G, hyper, src, nsteps)
        torch.cuda.synchronize()
        ctx["grad"] = L.grad.cpu().numpy().astype(np.float64)
        adv.copy_(keep)

    L._sgd_step = step
    _learn(L, _to_dev(r))
    torch.cuda.synchronize()
    assert ctx["step"] == w.STEPS and "grad" in ctx
    th0, klc = ctx["pre"]
    caught = []
    for p in range(w.P):
        rows = _step_rows(w, perms, p, target)
        e, _, _, msg, _ = grad_check(w, mode, ctx["grad"][p], th0[p], ctx["cols"], p, rows, klc[p], cfg)
        print(f"[D {w.name} {mode}: adv zeroed on the {n} rows of CTA {last}, step {target}, policy {p}] grad_err={e:.3g} "
              f"check: {'FAILED as required: ' + msg if msg else 'passed'}")
        caught.append(msg is not None)
    assert all(caught), f"B's check does not see the {n} rows of CTA {last}: {caught}"

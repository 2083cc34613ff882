"""N3 (SURVEY.md §8-f): RLlib 1.0.x checkpoint import / export without Ray — CPU tests on the committed golden fixtures
(tests/golden/ckpt_*.npz, extracted from the reference's own checkpoint files by tests/golden/make_golden.py)."""
import os
import pickle
import pickletools

import numpy as np
import pytest

from ddrl_b200 import checkpoint as C

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _from_golden(arch):
    z = np.load(os.path.join(GOLD, f"ckpt_{arch}.npz"), allow_pickle=True)
    from collections import OrderedDict
    pols = OrderedDict()
    for pid in [str(n) for n in z["names"]]:
        shapes = [tuple(int(x) for x in s if x > 0) for s in z[f"{pid}/shapes"]]
        pc = C.PolicyCheckpoint(theta=z[f"{pid}/theta"].copy(), shapes=shapes, filter_n=int(z[f"{pid}/filter_n"]),
                                filter_M=z[f"{pid}/filter_M"].copy(), filter_S=z[f"{pid}/filter_S"].copy(),
                                learner_stats={"cur_kl_coeff": 0.45, "cur_lr": 3e-4, "kl": 0.0141, "total_loss": 27.9})
        if f"{pid}/adam_m" in z.files:
            pc.adam_m, pc.adam_v = z[f"{pid}/adam_m"].copy(), z[f"{pid}/adam_v"].copy()
            pc.beta_powers = z[f"{pid}/beta_powers"].copy()
        pols[pid] = pc
    return C.Checkpoint(policies=pols, counters={"num_steps_sampled": 20000000, "num_steps_trained": 20000000})


def _assert_same(a: C.Checkpoint, b: C.Checkpoint):
    assert list(a.policies) == list(b.policies)
    assert a.counters == b.counters
    for pid in a.policies:
        x, y = a.policies[pid], b.policies[pid]
        assert np.array_equal(x.theta, y.theta) and x.theta.dtype == np.float32
        assert [tuple(s) for s in x.shapes] == [tuple(s) for s in y.shapes]
        assert x.filter_n == y.filter_n and np.array_equal(x.filter_M, y.filter_M) and np.array_equal(x.filter_S, y.filter_S)
        assert (x.adam_m is None) == (y.adam_m is None)
        if x.adam_m is not None:
            assert np.array_equal(x.adam_m, y.adam_m) and np.array_equal(x.adam_v, y.adam_v)
            assert np.array_equal(x.beta_powers, y.beta_powers)
        for k, v in x.learner_stats.items():
            assert y.learner_stats[k] == pytest.approx(v, rel=1e-7)


@pytest.mark.parametrize("arch", ["FullyDecentral", "Centralized", "TwoSides_TVel"])
def test_export_import_round_trip_is_bit_exact(arch, tmp_path):
    ck = _from_golden(arch)
    path = str(tmp_path / "checkpoint-1")
    C.save_rllib_checkpoint(path, ck)
    _assert_same(ck, C.load_rllib_checkpoint(path))
    pc = next(iter(ck.policies.values()))
    assert pc.theta.size == 128 * pc.obs_dim + 130 * pc.act_dim + 8513        # SURVEY.md §8 closed form


def test_exported_file_has_the_reference_schema(tmp_path):
    """Same nesting, key names / order and class paths as Results/**/checkpoint-1250 (SURVEY.md Appendix A)."""
    ck = _from_golden("FullyDecentral")
    path = str(tmp_path / "checkpoint-1")
    C.save_rllib_checkpoint(path, ck)
    import ddrl_b200.checkpoint as mod
    assert mod.MeanStdFilter.__module__ == "ddrl_b200.checkpoint"       # the temporary module patch was undone
    import sys
    assert "ray" not in sys.modules
    top = pickle.load(open(path, "rb"))                                 # the outer pickle holds plain types only
    assert set(top) == {"worker", "train_exec_impl"} and isinstance(top["worker"], bytes)
    assert set(top["train_exec_impl"]) == {"counters", "info", "timers"}
    globs = [arg for op, arg, _ in pickletools.genops(top["worker"]) if op.name in ("GLOBAL", "STACK_GLOBAL", "SHORT_BINUNICODE")
             and isinstance(arg, str)]
    assert "ray.rllib.utils.filter" in " ".join(globs) and "MeanStdFilter" in globs and "RunningStat" in globs
    ck2 = C.load_rllib_checkpoint(path)
    worker = C._StubUnpickler(__import__("io").BytesIO(top["worker"])).load()
    st = worker["state"]["policy_FL"]
    keys = list(st)
    assert keys[:4] == ["policy_FL/fc_1/kernel", "policy_FL/fc_1/bias", "policy_FL/fc_value_1/kernel", "policy_FL/fc_value_1/bias"]
    assert keys[-1] == "_optimizer_variables" and len(keys) == 13
    ov = list(st["_optimizer_variables"])
    assert ov[:4] == ["policy_FL/beta1_power", "policy_FL/beta2_power", "policy_FL/policy_FL/fc_1/kernel/Adam",
                      "policy_FL/policy_FL/fc_1/kernel/Adam_1"] and len(ov) == 26
    assert st["policy_FL/fc_1/kernel"].shape == (19, 64) and st["policy_FL/fc_out/kernel"].shape == (64, 4)
    f = worker["filters"]["policy_FL"]
    assert isinstance(f.rs._n, int) and f.rs._M.dtype == np.float64 and f.clip is None and f.demean and f.destd
    assert ck2.policies["policy_FL"].filter_n == 20020272                    # SURVEY.md Appendix A known answer


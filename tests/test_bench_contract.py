"""CPU: the reference arm of bench.py (the oracle port on the host cores) prints ONE JSON line with the contract's keys,
and the C-ABI header is plain C."""
import json
import os
import re
import shutil
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--envs", "32",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"].startswith("PPO learner agent-steps/sec") and d["unit"] == "agent-steps/s"
    for k in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
              "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert "workload" in d["config"] and "model" not in d["config"]
    # same-config contract: the reference arm describes its workload with the GPU arm's own config function
    sys.path.insert(0, ROOT)
    import bench
    assert d["config"] == bench.workload_config(32, 1, bench.WORKLOAD["minibatches_per_epoch"], 3)
    assert bench.workload_config(4096, 1, 32, 3)["envs_per_gpu"] == bench.WORKLOAD["envs_per_gpu"]   # default = configs[1]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["value"] > 0 and d["gpu_launches"] == 0


def test_reference_arm_other_ranks_exit_silently():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_every_supplementary_job_has_an_oracle_test(monkeypatch):
    """bench.run_supplementary's jobs, recorded without a GPU (time_fcnet / time_graphnet replaced by recorders), are the
    workload table of tests/test_gpu_supplementary_workloads.py plus the two jobs covered elsewhere: the fp32 job by the
    headline workload's fp32 mode, C4 by tests/test_gpu_graphnet_workload.py at its own envs and epochs."""
    import argparse
    import importlib
    sys.path.insert(0, ROOT)
    import bench
    from tests import test_gpu_bench_workload as H
    from tests import test_gpu_graphnet_workload as GN
    from tests import test_gpu_supplementary_workloads as S
    fc, gn = [], []
    monkeypatch.setattr(bench, "time_fcnet", lambda *a, **kw: fc.append((a, kw)) or {})
    monkeypatch.setattr(bench, "time_graphnet", lambda *a, **kw: gn.append((a, kw)) or (1.0, {"rows": 1}))
    out = bench.run_supplementary(argparse.Namespace(envs=4096, minibatches=32))
    assert not [v for v in out.values() if "error" in v], out
    jobs = dict(zip([k for k in out if k != "C4_shared_GraphNet"], fc))
    assert len(jobs) == len(fc) and set(out) == set(S.JOBS) | set(S.COVERED_ELSEWHERE)
    for name, (args, kw) in jobs.items():
        assert args[4:] == (3, 2) and not kw, (name, args, kw)           # steps, warmup as the table assumes
        if name in S.JOBS:
            assert args[:4] == S.JOBS[name], (name, args)
            assert name in S.EXPECT and name in S.IDS, name
    # the fp32 job: the headline's architecture and shape, which tests/test_gpu_bench_workload.py runs in its fp32 mode
    W = bench.WORKLOAD
    assert jobs["FullyDecentral_fp32_parity_kernel"][0][:4] == ("FullyDecentral", W["envs_per_gpu"], W["minibatches_per_epoch"], "fp32")
    assert H.MODES["fp32"]["mode"] == "fp32"
    # C4: time_graphnet(envs, epochs, steps, warmup) at the envs and epochs of the GraphNet workload test
    assert gn == [((4096, W["epochs"], 2, 1), {})], gn
    assert (GN.ENVS, GN.E_B) == gn[0][0][:2]
    for name, (module, test, param) in S.COVERED_ELSEWHERE.items():
        m = importlib.import_module(module)
        assert callable(getattr(m, test, None)), (name, module, test)
        assert param is None or param in m.MODES, (name, param)


@pytest.mark.skipif(shutil.which("gcc") is None, reason="gcc not available")
def test_header_is_plain_c():
    """include/ddrl_b200.h is the drop-in boundary: extern "C", plain pointers and sizes — it must compile as C99."""
    hdr = os.path.join(ROOT, "include", "ddrl_b200.h")
    out = subprocess.run(["gcc", "-std=c99", "-Wall", "-fsyntax-only", "-x", "c", hdr], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    code = re.sub(r"/\*.*?\*/", "", open(hdr).read(), flags=re.S)      # comments may mention torch; declarations may not
    assert "torch" not in code.lower() and "at::" not in code and "std::" not in code

"""bench.py --dump-outputs: the last timed learner iteration of the headline workload is written as float32 / float64 .npy
files (at most 64 MB); the same arguments give the same outputs, and --steps sets how many timed iterations ran."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SETS, WARMUP = 3, 1


def _bench_dump(out_dir, steps):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", str(WARMUP),
                        "--sets", str(SETS), "--no-cpu-baseline", "--no-supplementary", "--dump-outputs", str(out_dir)],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == steps
    files = sorted(os.listdir(out_dir))
    assert sum(os.path.getsize(os.path.join(out_dir, f)) for f in files) <= 64 << 20
    return {f[:-4]: np.load(os.path.join(out_dir, f)) for f in files}


def test_dump_outputs_are_reproducible_and_follow_steps(tmp_path):
    a = _bench_dump(tmp_path / "a", 2)
    b = _bench_dump(tmp_path / "b", 2)
    c = _bench_dump(tmp_path / "c", 3)
    assert {"theta", "adam_m", "adam_v", "filter_n", "logits", "value", "adv", "stats_total_loss"} <= set(a)
    assert set(a) == set(b) == set(c)
    for name, x in a.items():
        assert x.dtype in (np.float32, np.float64), name
        assert np.isfinite(x).all(), name
        assert np.array_equal(x, b[name]), name
    P, D = a["filter_M"].shape
    assert a["theta"].shape[0] == P and a["logits"].shape[0] == P and a["obs"].shape[2] == D
    # every learner iteration pushes its rollout rows through the filter: the dump must follow exactly the iterations up to
    # the last timed one (two untimed visits of every rollout set, the warm-up, the timed steps), not the e2e ones behind it
    sys.path.insert(0, ROOT)
    from bench import WORKLOAD as W
    rows = W["T"] * W["envs_per_gpu"] * (W["Ag"] // W["P"])
    for d, steps in ((a, 2), (c, 3)):
        assert (d["filter_n"] == (2 * SETS + WARMUP + steps) * rows).all(), (d["filter_n"], steps)
    assert not np.array_equal(a["theta"], c["theta"])

"""Device time of the learner's preparation phase with the two observation-filter modes, on the bench workload
(FullyDecentral: P = 4 policies, D = 19, A = 2, T = 32 steps x C = 4096 envs = 131 072 rows per policy, tensor-core
forward), alternated in one process with CUDA events (medians over rounds, after a warm-up of both):
  (a) the filter stage alone: `filter_update` (batch: push all rows, one normalisation table) against `filter_stream` +
      `filter_merge` (stream: row-by-row worker streams written as the obs column, W = 1 and 2 workers);
  (b) the whole preparation phase `FCNetLearner._prepare_cached` (filter, rollout + bootstrap forward, GAE, standardise,
      shuffle; replayed from its CUDA graph as learn_on_rollout runs it) in filter_mode "batch" and "stream";
  (c) the card name, power limit and SM clock, read in the same process.
The observations are 40 MB of float32 per call (fits in the 126 MB L2 after the first pass).
Usage: python tests/filter_stream_bench.py [--out FILE] [--rounds N] [--reps N]"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

P, D, A, T, C = 4, 19, 2, 32, 4096


def _time(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) * 1e3 / reps          # us per call


def _gpu_info():
    try:
        q = "name,power.limit,clocks.sm,clocks.max.sm"
        r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=60)
        return r.stdout.strip().splitlines()[torch.cuda.current_device()] if r.returncode == 0 else "nvidia-smi failed"
    except (OSError, subprocess.TimeoutExpired, IndexError):
        return "nvidia-smi unavailable"


def _alternate(fns, reps, rounds):
    for _ in range(3):
        for fn in fns.values():
            _time(fn, reps)
    t = {k: [] for k in fns}
    for _ in range(rounds):
        for k, fn in fns.items():
            t[k].append(_time(fn, reps))
    return {k: {"median_us": float(np.median(v)), "min_us": float(np.min(v)), "max_us": float(np.max(v))} for k, v in t.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=15)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    from ddrl_b200 import kernels as K
    from ddrl_b200.config import PPOConfig
    from ddrl_b200.learner import FCNetLearner
    from tests.util import ckpt_theta, synth_obs
    dev = torch.device("cuda")
    R = T * C
    theta, filt, _, _ = ckpt_theta("FullyDecentral")
    g = torch.Generator().manual_seed(0)
    raw = torch.from_numpy(synth_obs(filt, R, 1)).to(dev)                                   # [P, R, D]
    n0 = torch.tensor([f[0] for f in filt], dtype=torch.int64, device=dev)
    M0 = torch.from_numpy(np.stack([f[1] for f in filt])).to(dev)
    S0 = torch.from_numpy(np.stack([f[2] for f in filt])).to(dev)

    # (a) the filter stage alone (the state is restored from a copy before every call, so every call sees the same n)
    st = {k: v.clone() for k, v in (("n", n0), ("M", M0), ("S", S0))}
    norm = torch.empty(P, 2, D, dtype=torch.float64, device=dev)
    ws_b = torch.empty(K._lib.load().ddrl_filter_ws_bytes(P, R, D), dtype=torch.uint8, device=dev)
    out = torch.empty(P, R, D, device=dev)
    bufs = {W: (torch.empty(P, W, D, 3, dtype=torch.float64, device=dev),
                torch.empty(K.filter_stream_ws_bytes(P, T, C, W, D), dtype=torch.uint8, device=dev)) for W in (1, 2)}

    def reset():
        st["n"].copy_(n0), st["M"].copy_(M0), st["S"].copy_(S0)

    def batch():
        reset()
        K.filter_update(raw, st["n"], st["M"], st["S"], norm, ws_b)

    def stream(W):
        def f():
            reset()
            K.filter_stream(raw, st["n"], st["M"], st["S"], T, W, 0.0, out=out, parts=bufs[W][0], ws=bufs[W][1])
            K.filter_merge(bufs[W][0], R, st["n"], st["M"], st["S"], norm)
        return f

    def reset_only():
        reset()

    stage = _alternate({"reset": reset_only, "batch": batch, "stream_W1": stream(1), "stream_W2": stream(2)},
                       args.reps, args.rounds)

    # (b) the whole preparation phase, as learn_on_rollout runs it (CUDA-graph replay)
    rng = np.random.default_rng(2)
    raw4 = raw.reshape(P, T, C, D)
    boot = torch.from_numpy(synth_obs(filt, C, 3)).to(dev)
    rewards = torch.from_numpy((0.3 + 0.5 * rng.standard_normal((P, T, C))).astype(np.float32)).to(dev)
    dones = torch.from_numpy((rng.random((T, C)) < 1e-3).astype(np.uint8)).to(dev)
    eps = torch.randn(P, T, C, A, generator=g).to(dev)
    shuffle = torch.from_numpy(np.stack([rng.permutation(R) for _ in range(P)]).astype(np.int32)).to(dev)
    cfg = PPOConfig(num_sgd_iter=10, sgd_minibatch_size=R // 4)
    learners = {}
    for mode, W in (("batch", 1), ("stream", 1), ("stream", 2)):
        L = FCNetLearner(P, D, A, cfg, dev, theta=torch.from_numpy(theta), filter_mode=mode, filter_workers=W)
        b = L._alloc(T, C)
        obs_flat, eps_flat = raw4.reshape(P, R, D), eps.reshape(P, R, A)

        def prep(L=L, b=b, obs_flat=obs_flat, eps_flat=eps_flat):
            L._prepare_cached(b, obs_flat, boot, rewards, dones, eps_flat, shuffle, 1, True, T, C)
        prep(); prep()                      # eager first call, then the capture
        assert L._prep_graphs, getattr(L, "graph_error", None)
        learners[f"{mode}_W{W}"] = prep
    phase = _alternate(learners, max(1, args.reps // 4), args.rounds)
    res = {"workload": dict(P=P, D=D, A=A, T=T, C=C, rows_per_policy=R, obs_mb=P * R * D * 4 / 1e6),
           "gpu": _gpu_info(), "torch": torch.__version__, "filter_stage_us": stage, "prepare_phase_us": phase,
           "note": "filter_stage includes the state reset (3 small copies), timed alone as 'reset'"}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()

"""Cost of the leg coupling in the fused learner: SharedDecentralLegID (FCNet + LegCoupling, coupled SGD step) against
SharedDecentral (the same FCNet, D = 19, A = 2, uncoupled step) on the same resident inputs, alternated in one process.

Workload (the GraphNet supplementary shape): 4096 envs x 4 legs, T = 32 -> 524288 rows of ONE shared policy; E = 10 epochs
of 32 minibatches of 16384 rows; mode="tc" (one persistent launch per iteration), fixed-order reduction.
Prints agent-steps/s (rows per learner iteration over its time), us per optimizer step (iteration time / 320), and the card
and its power limit.  Usage: python tests/coupling_bench.py [--iters 6] [--out FILE]"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=6, help="timed iterations per variant (alternated)")
    ap.add_argument("--envs", type=int, default=4096)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("coupling_bench needs a CUDA device")
    from ddrl_b200.config import PPOConfig
    from ddrl_b200.learner import FCNetLearner
    import oracle.ddrl_oracle as O
    T, N, E, MB, D, A = 32, a.envs, 10, 16384, 19, 2
    C = 4 * N
    R = T * C
    nb = R // MB
    dev = "cuda"
    cfg = PPOConfig(num_sgd_iter=E, sgd_minibatch_size=MB)
    rng = np.random.default_rng(0)
    th = O.fcnet_init(D, 2 * A, torch.Generator().manual_seed(0))
    to = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(dev)
    raw = to((rng.standard_normal((1, T, C, D)) * 2 + 0.5).astype(np.float32))
    boot = to((rng.standard_normal((1, C, D)) * 2 + 0.5).astype(np.float32))
    rew = to((0.3 + 0.5 * rng.standard_normal((1, T, C))).astype(np.float32))
    dones = to((rng.random((T, N)) < 0.01).astype(np.uint8))
    eps = to(rng.standard_normal((1, T, C, A)).astype(np.float32))
    shuffle = to(rng.permutation(R).astype(np.int32)[None])
    perms = to(np.stack([rng.permutation(nb) for _ in range(E)]).astype(np.int32)[None])
    table = torch.tensor([0.7, -1.3, -0.4, 0.9, 1.6, -0.2, -1.1, 0.5])
    learners = {
        "SharedDecentralLegID (coupled)": FCNetLearner(1, D, A, cfg, dev, theta=torch.cat([th, table])[None],
                                                       leg_coupling=True, atomic_reduce=False),
        "SharedDecentral (uncoupled)": FCNetLearner(1, D, A, cfg, dev, theta=th[None], atomic_reduce=False),
    }
    times = {k: [] for k in learners}
    for L in learners.values():      # warm-up: module loads, graphs, buffers
        L.learn_on_rollout(raw, boot, rew, dones, eps, perms, shuffle=shuffle, cols_per_env=4)
    torch.cuda.synchronize()
    for _ in range(a.iters):
        for k, L in learners.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            L.learn_on_rollout(raw, boot, rew, dones, eps, perms, shuffle=shuffle, cols_per_env=4)
            torch.cuda.synchronize()
            times[k].append(time.perf_counter() - t0)
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                          text=True).stdout.strip()
    lines = [f"card: {card}",
             f"workload: {N} envs x 4 legs, T = {T} -> {R} rows, P = 1, E = {E}, {nb} minibatches of {MB}, mode=tc, "
             f"fixed-order reduction, {a.iters} alternated iterations per variant (median)"]
    med = {}
    for k, ts in times.items():
        m = float(np.median(ts))
        med[k] = m
        lines.append(f"{k:32s} {R / m / 1e6:8.2f} M agent-steps/s   {m / (E * nb) * 1e6:7.2f} us per optimizer step   "
                     f"(iterations: {', '.join(f'{t * 1e3:.2f}' for t in ts)} ms)")
    c, u = med["SharedDecentralLegID (coupled)"], med["SharedDecentral (uncoupled)"]
    lines.append(f"coupled / uncoupled iteration time: {c / u:.4f} ({(c / u - 1) * 100:+.2f} %)")
    txt = "\n".join(lines)
    print(txt)
    if a.out:
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()

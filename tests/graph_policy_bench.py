"""Device time of the shared GraphNet policy's sampler-side GPU work: ONE fused launch (`ddrl_graphnet_act`: forward +
DiagGaussian sample) against the two launches it replaces (`ddrl_graphnet_forward` under forward schedule 1, then
`ddrl_dg_sample`), alternated in one process with CUDA events, on the same resident inputs (ring graph, env-major legs):
  (a) compute_actions scale: B = 16 (4 envs x 4 legs) and B = 16 384 (4096 envs x 4 legs);
  (b) the forward + sample part of `GraphNetLearner.learn_on_rollout` at BASELINE.json configs[3]'s 524 288 rows
      (4096 envs x 4 legs x T = 32);
  (c) the card name and power limit, read in the same process.
The outputs of both variants are compared bit for bit at every size.  The working set of (a) fits in L2 (every rep re-reads
it from there); (b) streams 48 MB of state per call.  Usage: python tests/graph_policy_bench.py [--out FILE]"""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def _inputs(B, A, dev, g):
    from ddrl_b200.policies import QuantrupedDecentralizedSharedGraphEnv
    state = torch.randn(B, 4, 23, generator=g).to(dev)
    idx = torch.arange(4, dtype=torch.int32).repeat(B // 4).to(dev)
    adj = torch.from_numpy(QuantrupedDecentralizedSharedGraphEnv.create_adj()).float().expand(B, 4, 4).contiguous().to(dev)
    eps = torch.randn(B, A, generator=g).to(dev)
    return idx, state, adj, eps


def _time(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) * 1e3 / reps          # us per call


def compare(th, B, A, reps, rounds, dev, g):
    from ddrl_b200 import kernels as K
    idx, state, adj, eps = _inputs(B, A, dev, g)
    out2 = (torch.empty(B, 2 * A, device=dev), torch.empty(B, device=dev))
    out1 = (torch.empty(B, 2 * A, device=dev), torch.empty(B, device=dev), torch.empty(B, A, device=dev),
            torch.empty(B, device=dev))

    def two_launch():
        lg, v = K.graphnet_forward(th, idx, state, adj, A, out=out2)
        return (lg, v) + K.dg_sample(lg, eps)

    def fused():
        return K.graphnet_act(th, idx, state, adj, eps, A, out=out1)
    a, b = two_launch(), fused()
    torch.cuda.synchronize()
    identical = all(torch.equal(x, y) for x, y in zip(a, b))
    for _ in range(3):                                   # warm-up of both shapes
        _time(two_launch, reps)
        _time(fused, reps)
    t = {"two-launch": [], "fused": []}
    for _ in range(rounds):
        t["two-launch"].append(_time(two_launch, reps))
        t["fused"].append(_time(fused, reps))
    return identical, t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=15, help="alternated rounds per size")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("graph_policy_bench needs a CUDA device")
    from ddrl_b200 import kernels as K
    from ddrl_b200.modelv2 import _FlatParams, graphnet_shapes
    dev = torch.device("cuda", 0)
    A = 2
    g = torch.Generator().manual_seed(7)
    th = _FlatParams(graphnet_shapes(2 * A)).init_host(g, small=("actor/linear_out", "critic/linear_out")).to(dev)
    card = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    lines = [f"(c) card: {card}",
             f"A = {A}, ring graph, env-major legs; forward schedule 1; {a.rounds} alternated rounds per size, "
             "CUDA events around `reps` back-to-back calls; median (min .. max) us per call"]
    K.graphnet_set_variant(1)
    try:
        for tag, B, reps in (("(a) compute_actions, 4 envs x 4 legs", 16, 2000),
                             ("(a) compute_actions, 4096 envs x 4 legs", 16384, 200),
                             ("(b) learn_on_rollout forward + sample, configs[3]", 524288, 10)):
            identical, t = compare(th, B, A, reps, a.rounds, dev, g)
            med = {k: float(np.median(v)) for k, v in t.items()}
            lines.append(f"{tag}: B = {B}, {reps} calls per round, outputs bit-identical: {identical}")
            for k, v in t.items():
                lines.append(f"    {k:10s} {med[k]:10.2f} us  ({min(v):.2f} .. {max(v):.2f})")
            lines.append(f"    fused / two-launch: {med['fused'] / med['two-launch']:.4f}")
    finally:
        K.graphnet_set_variant(-1)
    txt = "\n".join(lines)
    print(txt)
    if a.out:
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()

"""Device time of the leg-coupled policy's inference (SharedDecentralLegID, model "cup" = FCNet + LegCoupling): ONE fused
launch (`ddrl_fcnet_forward_coupled` / `ddrl_fcnet_forward_tc_coupled`: forward + LegCoupling + DiagGaussian sample) against
the three launches it replaces (forward, `ddrl_leg_coupling`, `ddrl_dg_sample`), alternated in one process with CUDA events,
on the same resident inputs (D = 19, A = 2, node ids cycling over the four legs, MeanStdFilter normalisation):
  (a) FCNetLearner.compute_actions scale, FP32 entry: B = 16 (4 envs x 4 legs) and B = 16 384 (4096 envs x 4 legs);
  (b) the rollout forward of FCNetLearner._prepare, tensor-core entry, at 524 288 rows (4096 envs x 4 legs x T = 32);
  (c) the card name and power limit, read in the same process.
The outputs of both variants are compared bit for bit at every size.  The working set of (a) fits in L2; (b) streams
~40 MB of observations per call.  Usage: python tests/coupled_act_bench.py [--out FILE]"""
import argparse
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def _time(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) * 1e3 / reps          # us per call


def compare(kind, B, reps, rounds, dev, g):
    from ddrl_b200 import kernels as K
    import oracle.ddrl_oracle as O
    D, A = 19, 2
    theta = O.fcnet_init(D, 2 * A, torch.Generator().manual_seed(0)).float()[None].contiguous().to(dev)
    w = K.fcnet_tc_pack(theta, D, A) if kind == "tc" else theta
    obs = (torch.randn(1, B, D, generator=g) * 2 + 0.5).to(dev)
    norm = torch.stack([0.3 * torch.randn(D, generator=g), 1.0 / (0.2 + torch.rand(D, generator=g))]).double()[None].to(dev)
    node = (torch.arange(B, dtype=torch.int32) % 4)[None].contiguous().to(dev)
    eps = torch.randn(1, B, A, generator=g).to(dev)
    table = torch.tensor([[0.7, -1.3], [-0.4, 0.9], [1.6, -0.2], [-1.1, 0.5]]).to(dev)
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    mk = lambda: {"logits": torch.empty(1, B, 2 * A, device=dev), "value": torch.empty(1, B, device=dev),
                  "obs_out": torch.empty(1, B, D, device=dev)}
    o3, o1 = mk(), mk()
    o1.update(action=torch.empty(1, B, A, device=dev), logp=torch.empty(1, B, device=dev))
    act3, logp3 = torch.empty(B, A, device=dev), torch.empty(B, device=dev)
    from ddrl_b200 import _lib
    lib = _lib.load()

    def three_launch():
        if kind == "tc":
            K.fcnet_forward_tc(w, obs, A, norm=norm, out=o3, status=status)
        else:
            K.fcnet_forward(w, obs, A, norm=norm, out=o3)
        K.leg_coupling_(o3["logits"].view(B, 2 * A), node.view(B), table)
        _lib.check(lib.ddrl_dg_sample(o3["logits"].data_ptr(), eps.data_ptr(), B, A, act3.data_ptr(), logp3.data_ptr(),
                                      K._stream()), "dg_sample")

    def fused():
        f = K.fcnet_forward_tc_coupled if kind == "tc" else K.fcnet_forward_coupled
        f(w, obs, node, table, A, norm=norm, eps=eps, status=status, out=o1)

    three_launch()
    fused()
    torch.cuda.synchronize()
    identical = (all(torch.equal(o3[k], o1[k]) for k in ("logits", "value", "obs_out"))
                 and torch.equal(act3, o1["action"][0]) and torch.equal(logp3, o1["logp"][0]) and int(status.item()) == 0)
    for _ in range(3):                                   # warm-up of both variants
        _time(three_launch, reps)
        _time(fused, reps)
    t = {"three-launch": [], "fused": []}
    for _ in range(rounds):
        t["three-launch"].append(_time(three_launch, reps))
        t["fused"].append(_time(fused, reps))
    return identical, t


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=15, help="alternated rounds per size")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("coupled_act_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    g = torch.Generator().manual_seed(7)
    card = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    lines = [f"(c) card: {card}",
             f"D = 19, A = 2, filter normalisation on; {a.rounds} alternated rounds per size, CUDA events around `reps` "
             "back-to-back calls; median (min .. max) us per call"]
    for tag, kind, B, reps in (("(a) compute_actions, 4 envs x 4 legs, FP32", "fp32", 16, 2000),
                               ("(a) compute_actions, 4096 envs x 4 legs, FP32", "fp32", 16384, 200),
                               ("(b) _prepare rollout forward, 4096 envs x 4 legs x T = 32, tensor cores", "tc", 524288, 20)):
        identical, t = compare(kind, B, reps, a.rounds, dev, g)
        med = {k: float(np.median(v)) for k, v in t.items()}
        lines.append(f"{tag}: B = {B}, {reps} calls per round, outputs bit-identical: {identical}")
        for k, v in t.items():
            lines.append(f"    {k:12s} {med[k]:10.2f} us  ({min(v):.2f} .. {max(v):.2f})")
        lines.append(f"    fused / three-launch: {med['fused'] / med['three-launch']:.4f}")
    txt = "\n".join(lines)
    print(txt)
    if a.out:
        with open(a.out, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main()

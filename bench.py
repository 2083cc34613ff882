#!/usr/bin/env python
"""Benchmark of the DDRL learner hot path on B200 (contract: see the task statement / DESIGN.md §Measurement).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" is ONE learner iteration of the BASELINE.json configs[1] workload
(FullyDecentral: 4 per-leg FCNet policies 19->2, 4096 parallel envs per GPU, fragment T=32, 10 SGD epochs):
filter update+normalise -> forward/sample/logp/value -> bootstrap -> GAE -> standardise -> shuffle ->
10 x 32 minibatch steps (fused fwd + PPO loss + bwd, gradient reduce, [NCCL all-reduce], clip + TF1 Adam)
-> KL-coefficient update.  Metric: agent-steps/s = T * envs * agents / time, whole job over all ranks.
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOAD = dict(name="FullyDecentral (BASELINE.json configs[1])", P=4, Ag=4, D=19, A=2, envs_per_gpu=4096, T=32,
                epochs=10, minibatches_per_epoch=32)
METRIC = "PPO learner agent-steps/sec (fwd+GAE+update)"
UNIT = "agent-steps/s"


def workload_config(envs, world, nb, sets):
    """The workload description both arms print as `config` (identical dicts at the same --gpus / --envs / --minibatches)."""
    W = WORKLOAD
    C = envs * (W["Ag"] // W["P"])
    R = W["T"] * C
    return {"workload": W["name"], "policies": W["P"], "agents_per_env": W["Ag"], "obs_dim": W["D"], "act_dim": W["A"],
            "envs_per_gpu": envs, "envs_total": envs * world, "fragment_T": W["T"], "rows_per_policy_per_gpu": R,
            "num_sgd_iter": W["epochs"], "minibatches_per_epoch": nb, "sgd_minibatch_size_global": (R // nb) * world,
            "inputs": f"{sets} rotating synthetic rollout sets per GPU (seeds 1234 + rank + 100 * set), visited round robin: "
                      "the sets exceed the 126 MB L2 in aggregate, no explicit flush"}


def flops_per_agent_step(D, A, E):
    """SURVEY.md §8-d: MACs = (1+3E)*F - 128*E*D, F = 128D + 128A + 8256; flops = 2x."""
    F = 128 * D + 128 * A + 8256
    return 2 * ((1 + 3 * E) * F - 128 * E * D)


def train_flops_per_row(D, A):
    F = 128 * D + 128 * A + 8256
    return 2 * (3 * F - 128 * D)


# ------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md clocks line)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc, self.t0, self.t1 = index, [], None, None, None

    def start(self, wait_first=10.0):
        """Spawn `nvidia-smi -lms 100` and wait for its FIRST sample: NVML initialisation takes 50-500 ms and stalls CUDA
        calls of the process meanwhile — started right in front of the warm-up it used to land inside the timed region of
        short runs (10-60 ms hiccups in 3 of 9 five-step runs).  Sampling itself goes on through the timed region."""
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
            t_end = time.time() + wait_first
            while not self.rows and time.time() < t_end and self.proc.poll() is None:
                time.sleep(0.01)
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def mark(self, begin):
        """Host time stamps of the timed region (set right after / before the synchronising barriers)."""
        if begin:
            self.t0 = time.time()
        else:
            self.t1 = time.time()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = self.rows
        if self.t0 is not None and self.t1 is not None:      # samples taken while the timed region ran (+ one period)
            inside = [r for r in rows if self.t0 <= r[0] <= self.t1 + 0.1]
            rows = inside or rows
        sm, mx, reasons = [], None, set()
        for _, r in rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------
def synth_rollout(P, T, C, D, A, envs, nb, E, seed, device=None, pinned=False):
    """Synthetic quantruped-shaped rollout (SURVEY.md §8-d): raw obs ~ N(mu_k, sigma_k^2) with per-feature scales
    spanning 0.1..89 like the FullyDecentral checkpoint filter, rewards ~ N(0.3, 0.5^2), done ~ Bernoulli(1e-3)."""
    import torch
    g = torch.Generator().manual_seed(seed)
    mu = torch.linspace(-0.5, 3.0, D)
    sigma = torch.logspace(-1.0, 1.95, D)
    raw = mu + sigma * torch.randn(P, T, C, D, generator=g)
    boot = mu + sigma * torch.randn(P, C, D, generator=g)
    rewards = 0.3 + 0.5 * torch.randn(P, T, C, generator=g)
    dones = (torch.rand(T, envs, generator=g) < 1e-3).to(torch.uint8)
    eps = torch.randn(P, T, C, A, generator=g)
    perms = torch.stack([torch.stack([torch.randperm(nb, generator=g) for _ in range(E)]) for _ in range(P)]).int()
    shuffle = torch.stack([torch.randperm(T * C, generator=g) for _ in range(P)]).int()
    out = dict(raw=raw.float(), boot=boot.float(), rewards=rewards.float(), dones=dones, eps=eps.float(), perms=perms,
               shuffle=shuffle)
    if pinned:
        out = {k: v.contiguous().pin_memory() for k, v in out.items()}
    if device is not None:
        out = {k: v.to(device) for k, v in out.items()}
    return out


class CpuLearner:
    """The oracle's float32 torch twin (CPU restatement of the reference's TF-CPU learner iteration: RLlib 1.0.1 around the
    reference's models) with persistent policy state, on `envs` environments of the workload (same P/D/A/T/E and
    minibatches per epoch).  The P policies are independent, so they run on P host threads, each with cores/P intra-op
    threads (measured faster than one policy at a time with all cores: the matrices are small)."""

    def __init__(self, envs, nb=None, threads=None):
        import torch
        import oracle.ddrl_oracle as O
        self.O, self.torch = O, torch
        W = WORKLOAD
        self.P, self.D, self.A, self.T, self.E = W["P"], W["D"], W["A"], W["T"], W["epochs"]
        self.nb = nb or W["minibatches_per_epoch"]
        self.envs, self.Ag = envs, W["Ag"]
        self.C = envs * (W["Ag"] // self.P)
        self.threads = threads or os.cpu_count() or 1
        self.par = self.P if self.threads >= 2 * self.P else 1
        torch.set_num_threads(max(1, self.threads // self.par))
        self.cfg = O.PPOConfig(num_sgd_iter=self.E, sgd_minibatch_size=(self.T * self.C) // self.nb)
        gen = torch.Generator().manual_seed(1234)
        self.pols = [O.PolicyState(O.fcnet_init(self.D, 2 * self.A, gen),
                                   O.AdamState.zeros(O.n_params(O.fcnet_shapes(self.D, 2 * self.A)), torch.float32, self.cfg),
                                   O.MeanStdFilter((self.D,), clip=None), self.cfg.kl_coeff) for _ in range(self.P)]

    def rollout(self, seed):
        r = synth_rollout(self.P, self.T, self.C, self.D, self.A, self.envs, self.nb, self.E, seed)
        return {k: v.numpy() for k, v in r.items()}

    def iteration(self, r):
        """One learner iteration on rollout set r -> seconds."""
        O, A, cfg = self.O, self.A, self.cfg

        def one(p):
            sl = slice(p, p + 1)
            return O.fcnet_learner_iteration(self.pols[sl], r["raw"][sl], r["boot"][sl], r["rewards"][sl], r["dones"], r["eps"][sl],
                                             r["shuffle"][sl], r["perms"][sl], 2 * A, cfg, self.torch.float32)
        t0 = time.perf_counter()
        if self.par > 1:
            from concurrent.futures import ThreadPoolExecutor
            with ThreadPoolExecutor(self.par) as ex:
                list(ex.map(one, range(self.P)))
        else:
            for p in range(self.P):
                one(p)
        return time.perf_counter() - t0

    def agent_steps(self):
        return self.T * self.envs * self.Ag


def cpu_iteration_baseline(envs, seed=0, threads=None):
    """One CPU learner iteration on a bounded sample (`envs` environments) -> (agent-steps/s, seconds, threads)."""
    L = CpuLearner(envs, threads=threads)
    dt = L.iteration(L.rollout(seed))
    return L.agent_steps() / dt, dt, L.threads


# ------------------------------------------------------------------------------------------------------------
def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path, on OUR arm's config (same envs per GPU, T,
    epochs, minibatches; the same rotating synthetic rollout sets).  TF/Ray cannot be installed here (DESIGN.md §6), so
    this times the oracle port (float32 torch twin of the RLlib 1.0.1 learner iteration) with all host threads.  Under
    torchrun rank 0 alone runs it (one GPU's share of the workload: the metric is per-job agent-steps/s of the CPU path)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    os.environ.pop("OMP_NUM_THREADS", None)      # torchrun pins it to 1: the CPU arm may use every host core
    W = WORKLOAD
    envs, nb = args.envs, args.minibatches
    L = CpuLearner(envs, nb=nb, threads=os.cpu_count() or 1)
    sets = [L.rollout(1234 + 100 * s_) for s_ in range(args.sets)]
    times = []
    for i in range(args.warmup + args.steps):
        dt = L.iteration(sets[i % len(sets)])
        if i >= args.warmup:
            times.append(dt)
    ms = float(np.mean(times) * 1e3)
    value = L.agent_steps() / (ms * 1e-3)
    sample = (f"all {envs} envs x T={W['T']} x {W['Ag']} agents per step (the full per-GPU workload of the GPU arm), "
              f"{L.par} policy threads x {max(1, L.threads // L.par)} intra-op threads")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(envs, 1, nb, args.sets),
        "note": "oracle port (torch CPU float32 twin of the RLlib 1.0.1 learner iteration); TF/Ray are not installable offline; "
                "one GPU's share of the workload on the host cores whatever --gpus says",
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": L.threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


DUMP_ROWS = 32768      # rows per policy kept of the per-row outputs: a fixed, seeded sample when the rollout has more


def dump_outputs(out_dir, L, stats):
    """--dump-outputs: what one FCNetLearner.learn_on_rollout call gave its caller, as out_dir/<name>.npy in float32 / float64:
    the per-policy stats it returned (stats_<key>), the state it left (weights, Adam moments and beta powers, observation
    filter, KL coefficient) and the per-row outputs of its forward pass and GAE in rollout order (filtered observations,
    actions, logits, log-probabilities, values, standardised advantages, value targets; the same DUMP_ROWS rows of every
    policy when the rollout has more).  The inputs depend on the arguments alone, and so do the outputs, except with
    --atomic-reduce."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    arrays = {f"stats_{k}": np.array([s[k] for s in stats], dtype=np.float64) for k in stats[0]}
    arrays.update(theta=L.theta, adam_m=L.m, adam_v=L.v, adam_beta_pow=L.beta_pow, kl_coeff=L.kl_coeff,
                  filter_n=L.filt_n, filter_M=L.filt_M, filter_S=L.filt_S)
    b = L._bufs
    R = b["value"].shape[1]
    rows = np.arange(R) if R <= DUMP_ROWS else np.sort(np.random.default_rng(0).choice(R, DUMP_ROWS, replace=False))
    rows = torch.from_numpy(rows).to(L.device)
    for name in ("obs", "act", "logits", "logp", "value", "adv", "vtarg"):
        arrays[name] = b[name].index_select(1, rows)
    for name, a in arrays.items():
        a = a.cpu().numpy() if torch.is_tensor(a) else a
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64 if a.dtype in (np.float64, np.int64) else np.float32))


def time_graphnet(envs, epochs, steps, warmup, step_kind="tc"):
    """BASELINE.json configs[3] — shared GraphNet policy over the 4-leg graph, `envs` envs x 4 agents, T=32, one weight set,
    minibatch = rows/32; -> (ms per learner iteration, config dict)."""
    import torch
    from ddrl_b200.config import PPOConfig
    from ddrl_b200.learner import GraphNetLearner
    from ddrl_b200.modelv2 import _FlatParams, graphnet_shapes
    from ddrl_b200.policies import QuantrupedDecentralizedSharedGraphEnv
    dev = torch.device("cuda", torch.cuda.current_device())
    A, T, N, E = 2, 32, envs, epochs
    C, R = N * 4, T * N * 4
    nb = 32
    cfg = PPOConfig(num_sgd_iter=E, sgd_minibatch_size=R // nb)
    g = torch.Generator().manual_seed(7)
    th = _FlatParams(graphnet_shapes(2 * A)).init_host(g, small=("actor/linear_out", "critic/linear_out")).reshape(1, -1)
    L = GraphNetLearner(A, cfg, dev, theta=th, step=step_kind)
    state = torch.randn(T, C, 4, 23, generator=g).to(dev)
    idx = torch.arange(4, dtype=torch.int32).repeat(T * N).reshape(T, C).to(dev)
    adj = torch.from_numpy(QuantrupedDecentralizedSharedGraphEnv.create_adj()).float().expand(T, C, 4, 4).contiguous().to(dev)
    rewards = (0.3 + 0.5 * torch.randn(T, C, generator=g)).to(dev)
    dones = (torch.rand(T, N, generator=g) < 1e-3).to(torch.uint8).to(dev)
    eps = torch.randn(T, C, A, generator=g).to(dev)
    perms = torch.stack([torch.randperm(nb, generator=g) for _ in range(E)]).int().to(dev)
    shuffle = torch.randperm(R, generator=g).int().to(dev)

    def step():
        return L.learn_on_rollout(idx, state, adj, idx[0], state[0], adj[0], rewards, dones, eps, perms, shuffle)
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    return ms, {"workload": "Shared GraphNet policy over the 4-leg graph (BASELINE.json configs[3])", "envs": N, "fragment_T": T,
                "rows": R, "num_sgd_iter": E, "minibatches_per_epoch": nb, "sgd_step": L.step_kind}


def run_graphnet(args):
    """Supplementary line (not the headline): BASELINE.json configs[3]."""
    import torch
    torch.cuda.set_device(0)
    ms, cfgd = time_graphnet(args.envs, args.gn_epochs, args.steps, args.warmup, args.gn_step)
    print(json.dumps({"metric": METRIC, "value": cfgd["rows"] / (ms * 1e-3), "unit": UNIT, "n_gpus": 1, "steps": args.steps,
                      "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "dtype": "f32", "data": "synthetic",
                      "config": dict(cfgd, note="supplementary")}))


def time_fcnet(arch, envs, nb, mode, steps, warmup, sets=2):
    """A short resident-input timing of one architecture / shape on the current device (same harness as the headline, fewer
    steps) -> dict(agent-steps/s, ms per iteration, us per optimizer step)."""
    import torch
    from ddrl_b200.config import PPOConfig
    from ddrl_b200.learner import FCNetLearner
    from ddrl_b200.modelv2 import fcnet_init_flat
    from ddrl_b200.policies import ARCHITECTURES
    tvel = arch.endswith("_TVel")
    env = ARCHITECTURES["QuantrupedMultiEnv_" + arch.replace("_TVel", "")]
    P, Ag, D, A = len(env.policy_names), len(env.agent_names), env.obs_dim(tvel), env.act_dim()
    T, E = WORKLOAD["T"], WORKLOAD["epochs"]
    dev = torch.device("cuda", torch.cuda.current_device())
    C = envs * (Ag // P)
    R = T * C
    cfg = PPOConfig(num_sgd_iter=E, sgd_minibatch_size=R // nb)
    gen = torch.Generator().manual_seed(1234)
    L = FCNetLearner(P, D, A, cfg, dev, theta=torch.stack([fcnet_init_flat(D, 2 * A, gen) for _ in range(P)]), mode=mode)
    rs = [synth_rollout(P, T, C, D, A, envs, nb, E, 77 + s_, device=dev) for s_ in range(sets)]

    def step(i):
        r = rs[i % sets]
        return L.learn_on_rollout(r["raw"], r["boot"], r["rewards"], r["dones"], r["eps"], r["perms"], r["shuffle"])
    # the first call runs the preparation phase eagerly, every later call captures the CUDA graph of its rollout set on first
    # sight: sets + 1 untimed calls leave no capture inside the timed region (with warmup = sets the third call — the first
    # TIMED one — used to capture set 0: several ms in a 3-step measurement)
    warmup = max(warmup, sets + 1)
    for i in range(warmup):
        step(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        step(warmup + i)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    # the SGD phase alone: E launches (persistent) or E * nb steps
    b = L._bufs
    src = {n_: b[n_ + "_s"] for n_ in ("obs", "act", "logits", "logp", "value", "adv", "vtarg")}
    MB, _, G = L._sgd_setup(R)
    hyper = L._hyper(MB)
    pers = L._persistent_steps(G)
    L.step_ctr.zero_()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    nl = 2 if pers else min(E * nb, 64)
    e0.record()
    for _ in range(nl):
        if pers:
            L.step_ctr.zero_()
        L._sgd_step(b, MB, G, hyper, src, nsteps=E * nb if pers else 1)
    e1.record()
    torch.cuda.synchronize()
    us_step = 1e3 * e0.elapsed_time(e1) / (nl * (E * nb if pers else 1))
    del L, rs
    return {"arch": arch, "policies": P, "agents_per_env": Ag, "obs_dim": D, "act_dim": A, "envs": envs, "rows_per_policy": R,
            "minibatches_per_epoch": nb, "sgd_minibatch_size": R // nb, "mode": mode, "value": T * envs * Ag / (ms * 1e-3),
            "unit": UNIT, "ms_per_step": ms, "us_per_sgd_step": us_step, "steps": steps, "warmup": warmup}


def run_supplementary(args):
    """Short resident-input runs of the other BASELINE.json configs (3 timed iterations each after 2 warm-ups; the headline
    stays configs[1]): C1 the reference's own latency-bound minibatch shape, Local, Centralized, the FP32-parity SGD kernel
    and the shared GraphNet policy at the configured 10 epochs."""
    import torch
    out = {}
    jobs = [("C1_reference_minibatch_shape_FullyDecentral_16000rows_MB128", ("FullyDecentral", 500, 125, "tc")),
            ("C1_Centralized_16000rows_MB128", ("Centralized", 500, 125, "tc")),
            ("C3_Local", ("Local", args.envs, args.minibatches, "tc")),
            ("Centralized", ("Centralized", args.envs, args.minibatches, "tc")),
            ("FullyDecentral_fp32_parity_kernel", ("FullyDecentral", args.envs, args.minibatches, "fp32"))]
    for name, (arch, envs, nb, mode) in jobs:
        try:
            out[name] = time_fcnet(arch, envs, nb, mode, 3, 2)
        except Exception as exc:      # supplementary only: never lose the headline line
            out[name] = {"error": repr(exc)}
        torch.cuda.empty_cache()
    try:
        ms, cfgd = time_graphnet(args.envs, WORKLOAD["epochs"], 2, 1)
        out["C4_shared_GraphNet"] = dict(cfgd, value=cfgd["rows"] / (ms * 1e-3), unit=UNIT, ms_per_step=ms, steps=2, warmup=1)
    except Exception as exc:
        out["C4_shared_GraphNet"] = {"error": repr(exc)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs", type=int, default=WORKLOAD["envs_per_gpu"], help="envs per GPU")
    ap.add_argument("--minibatches", type=int, default=WORKLOAD["minibatches_per_epoch"])
    ap.add_argument("--cpu-envs", type=int, default=1024, help="envs in the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-supplementary", action="store_true", help="skip the short supplementary runs of the other BASELINE configs")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--mode", default="tc", choices=["tc", "fp32"], help="SGD-step kernel: tcgen05 split-fp16 or FP32 FMA")
    ap.add_argument("--tc-variant", type=int, default=0, choices=[0, 1, 2],
                    help="tcgen05 schedule: 0 auto, 1 branch-sequential, 2 ping-pong (A/B timing)")
    ap.add_argument("--ctas", type=int, default=0, help="CTAs per policy of the SGD-step kernel (0 = the learner's choice)")
    ap.add_argument("--sets", type=int, default=3, help="rotating rollout sets (aggregate > L2)")
    ap.add_argument("--gn-step", default="tc", choices=["tc", "three-kernel", "two-launch"],
                    help="graphnet workload: SGD-step kernel (tc = persistent tensor-core step, default)")
    ap.add_argument("--workload", default="fcnet", choices=["fcnet", "graphnet"])
    ap.add_argument("--arch", default="FullyDecentral",
                    help="supplementary: any published architecture (Centralized, FullyDecentral, Local, SingleNeighbor, "
                         "SingleDiagonal, SingleToFront, TwoSides, TwoDiags; append _TVel for the target-velocity obs); "
                         "the headline line is the default FullyDecentral = BASELINE.json configs[1]")
    ap.add_argument("--gn-epochs", type=int, default=WORKLOAD["epochs"])
    ap.add_argument("--atomic-reduce", action="store_true",
                    help="tc SGD step: add the per-CTA partial gradients into FCNetLearner's L2 accumulation vector (float "
                         "atomics, the library default) instead of summing them in a fixed order; faster, but the order of "
                         "the additions changes from run to run and so do the results (profiles/r03_reduction_reproducibility.txt)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed learner iteration computed as DIR/<name>.npy (same arguments, same inputs)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.workload != "fcnet"):
        ap.error("--dump-outputs: only the FCNet workload of --impl ours")
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.arch != "FullyDecentral":      # supplementary architectures: same harness, the architecture's P / D / A
        from ddrl_b200.policies import ARCHITECTURES
        tvel = args.arch.endswith("_TVel")
        env = ARCHITECTURES["QuantrupedMultiEnv_" + args.arch.replace("_TVel", "")]
        if len(env.agent_names) != len(env.policy_names):
            raise SystemExit("--arch: only the published one-agent-per-policy architectures")
        WORKLOAD.update(name=f"{args.arch} (supplementary architecture, same harness as configs[1])", P=len(env.policy_names),
                        Ag=len(env.agent_names), D=env.obs_dim(tvel), A=env.act_dim())
    if args.impl == "reference":
        return run_reference(args)
    if args.workload == "graphnet":
        return run_graphnet(args)

    import torch
    import torch.distributed as dist
    from ddrl_b200 import kernels as K
    from ddrl_b200.config import PPOConfig
    from ddrl_b200.learner import FCNetLearner

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # stdout carries exactly ONE JSON line: anything libraries print meanwhile (NCCL's version banner) goes to stderr
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus or world == 1, f"--gpus {args.gpus} but WORLD_SIZE={world}"

    W = WORKLOAD
    P, D, A, T, E, Ag = W["P"], W["D"], W["A"], W["T"], W["epochs"], W["Ag"]
    envs = args.envs
    C = envs * (Ag // P)
    R = T * C
    nb = args.minibatches
    MB_local = R // nb
    cfg = PPOConfig(num_sgd_iter=E, sgd_minibatch_size=MB_local * world)

    if args.tc_variant:
        K.tc_set_variant(args.tc_variant)
    if os.environ.get("DDRL_TC_CLUSTER"):      # A/B switch: thread-block cluster size of the ping-pong kernel (default off)
        K.tc_set_cluster(int(os.environ["DDRL_TC_CLUSTER"]))
    from ddrl_b200.modelv2 import fcnet_init_flat      # the product's own GlorotUniformScaled initialiser
    gen = torch.Generator().manual_seed(1234)
    theta0 = torch.stack([fcnet_init_flat(D, 2 * A, gen) for _ in range(P)])
    # the fixed-order reduction of the partial gradients by default: with the same arguments every run computes the same
    # results, so the outputs of two builds can be compared (--dump-outputs)
    L = FCNetLearner(P, D, A, cfg, dev, theta=theta0, use_graph=not args.no_graph, mode=args.mode,
                     ctas_per_policy=args.ctas or None, atomic_reduce=args.atomic_reduce)

    sets = [synth_rollout(P, T, C, D, A, envs, nb, E, 1234 + rank + 100 * s, device=dev) for s in range(args.sets)]
    host = {k: v.contiguous().pin_memory() for k, v in synth_rollout(P, T, C, D, A, envs, nb, E, 999 + rank).items()
            if k in ("rewards", "dones", "perms", "shuffle")}   # pinned e2e inputs besides the observations (below)
    bytes_per_set = sum(v.numel() * v.element_size() for v in sets[0].values())

    def step_resident(i):
        s = sets[i % len(sets)]
        return L.learn_on_rollout(s["raw"], s["boot"], s["rewards"], s["dones"], s["eps"], s["perms"], s["shuffle"])

    # e2e inputs arrive the way the reference's env produces them: ONE full 43-dim observation per env step (pinned host
    # memory); the per-agent index gather (distribute_observations / get_obs_indices) runs on the device (ddrl_obs_gather,
    # bit-exact), so the H2D copy carries 43 floats per env step instead of P x D gathered ones
    from ddrl_b200.policies import ARCHITECTURES
    arch_env = ARCHITECTURES["QuantrupedMultiEnv_" + args.arch.replace("_TVel", "")]
    tvel = args.arch.endswith("_TVel")
    table = torch.from_numpy(arch_env.gather_table(tvel)).to(dev)
    Dfull = 43 + int(tvel)
    gfull = torch.Generator().manual_seed(4242 + rank)
    mu_f, sg_f = torch.linspace(-0.5, 3.0, Dfull), torch.logspace(-1.0, 1.95, Dfull)
    host_full = (mu_f + sg_f * torch.randn(T * envs, Dfull, generator=gfull)).float().contiguous().pin_memory()
    host_boot = (mu_f + sg_f * torch.randn(envs, Dfull, generator=gfull)).float().contiguous().pin_memory()
    host_small = host
    draw = torch.empty(P, T * C, D, dtype=torch.float32, device=dev)
    dbootg = torch.empty(P, C, D, dtype=torch.float32, device=dev)
    h2d = sum(v.numel() * v.element_size() for v in list(host_small.values()) + [host_full, host_boot])
    # double-buffered input staging: the H2D copy of step i+1 runs on a copy stream while step i computes (every step's
    # copy is inside the timed region; the step waits for its own copy before it touches the data)
    copy_stream = torch.cuda.Stream(device=dev)
    stage = [dict(full=torch.empty_like(host_full, device=dev), boot=torch.empty_like(host_boot, device=dev),
                  small={k: torch.empty_like(v, device=dev) for k, v in host_small.items()},
                  ready=torch.cuda.Event(), free=torch.cuda.Event()) for _ in range(2)]
    state = {"next": 0, "primed": False}
    eps_buf = torch.empty(P, T, C, A, device=dev)

    def enqueue_copy(slot):
        s = stage[slot]
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(s["free"])           # the compute that last read this slot is done
            s["full"].copy_(host_full, non_blocking=True)
            s["boot"].copy_(host_boot, non_blocking=True)
            for k, v in s["small"].items():
                v.copy_(host_small[k], non_blocking=True)
            s["ready"].record(copy_stream)

    def step_e2e(i):
        cur = torch.cuda.current_stream(dev)
        if not state["primed"]:
            for s in stage:
                s["free"].record(cur)
            enqueue_copy(0)
            state["primed"] = True
        slot = state["next"]
        s = stage[slot]
        enqueue_copy(1 - slot)                          # prefetch the next step's inputs behind this step's compute
        state["next"] = 1 - slot
        cur.wait_event(s["ready"])
        K.obs_gather(s["full"], table, P, out=draw)
        K.obs_gather(s["boot"], table, P, out=dbootg)
        eps_buf.normal_()                               # fresh sampling noise, generated on the device
        out = L.learn_on_rollout(draw.view(P, T, C, D), dbootg, s["small"]["rewards"], s["small"]["dones"], eps_buf,
                                 s["small"]["perms"], s["small"]["shuffle"])   # host floats: includes the D2H read of the stats
        s["free"].record(cur)
        return out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    last = {}

    def timed(fn, warmup, steps, sampler=None):
        for i in range(warmup):
            fn(i)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if sampler is not None:
            sampler.mark(True)
        e0.record()
        for i in range(steps):
            last["out"] = fn(warmup + i)
        e1.record()
        barrier()
        if sampler is not None:
            sampler.mark(False)
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # one-time setup, not a warm-up step of the contract: the learner runs its first call eagerly and captures the preparation
    # phase into a CUDA graph at the first REPLAYED use of each set of input buffers (capture = synchronize + ~3-15 ms).  With
    # 3 rotating sets and W = 3 the third capture used to fall on the first TIMED step; every set is visited twice here so that
    # the W warm-up steps and the K timed steps are all steady-state iterations.
    for j in range(2 * len(sets)):
        step_resident(j)
    barrier()
    clocks = ClockSampler(local)
    n0 = K.launch_count()
    clocks.start()
    ms_total = timed(step_resident, args.warmup, args.steps, clocks)
    clk = clocks.stop()
    if args.dump_outputs:      # before the e2e and kernel timings below move the learner on
        if rank == 0:
            dump_outputs(args.dump_outputs, L, last["out"])
        barrier()
    # kernels per iteration: API launches outside the captured graph + graph replays x nodes
    steps_per_iter = E * nb
    G_ = L._sgd_setup(R)[2]
    fused = L.fuse_tail and G_ * P <= L.sms     # train kernel carries reduce + [peer all-reduce] + clip + Adam
    per_sgd = 1 if fused else 3
    sgd_launches = 1 if L._persistent_steps(G_) else steps_per_iter * per_sgd    # persistent: ONE launch for all E * nb steps
    launches_per_iter = 1 + 2 + 2 + 2 + 1 + 7 + sgd_launches   # pack, filter x2, fwd x2, gae x2, standardise, 7 gathers, sgd
    ms_e2e = timed(step_e2e, max(4, args.warmup), max(3, args.steps // 2))   # warm-up covers both staging slots (graph capture)
    e2e_steps = max(3, args.steps // 2)

    agent_steps = T * envs * Ag * world
    value = agent_steps * args.steps / (ms_total * 1e-3)
    e2e_value = agent_steps * e2e_steps / (ms_e2e * 1e-3)

    # ---- roofline of the dominant kernel: the SGD-step kernel exactly as the product path launches it (fused forward +
    # PPO loss + backward + gradient reduce + [peer all-reduce] + clip + Adam; persistent: one launch = the E * nb steps of
    # an iteration), each launch bracketed by CUDA events on the launching (= torch current) stream -------------------------
    b = L._bufs
    src = {n_: b[n_ + "_s"] for n_ in ("obs", "act", "logits", "logp", "value", "adv", "vtarg")}
    MB, nbb, G = L._sgd_setup(R)
    hyper = L._hyper(MB * world)
    persistent = L._persistent_steps(G)
    steps_per_launch = E * nb if persistent else 1      # as the product path launches it: all steps of an iteration
    n_launch = 5 if persistent else 40
    evs = []
    L.step_ctr.zero_()
    barrier()
    for i in range(n_launch):
        a, c = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if persistent:
            L.step_ctr.zero_()      # every launch runs steps 0 .. E * nb - 1 of the minibatch schedule
        a.record()
        L._sgd_step(b, MB, G, hyper, src, nsteps=steps_per_launch)
        c.record()
        evs.append((a, c))
    torch.cuda.synchronize()
    k_ms = float(np.mean([a.elapsed_time(c) for a, c in evs[1 if persistent else 2:]]))
    flops_launch = train_flops_per_row(D, A) * MB * P * steps_per_launch
    achieved_tf = flops_launch / (k_ms * 1e-3) / 1e12
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    tensor_peak = float(peaks.get("bf16_tflops_sustained", 1400.0))
    # DRAM traffic of that kernel: read from the committed ncu artefact of the same launch shape (never a constant here)
    traffic, traffic_note = None, "no ncu --set full capture of this launch shape under profiles/"
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        for ent in tr["captures"]:
            c = ent["shape"]
            if (c["arch"] == args.arch and c["envs_per_gpu"] == envs and c["minibatches_per_epoch"] == nb and c["mode"] == args.mode
                    and c["sgd_steps_per_launch"] == steps_per_launch and c["world"] == world):
                traffic = float(ent["dram_bytes_read"]) + float(ent["dram_bytes_write"])
                traffic_note = f"dram__bytes_read.sum + dram__bytes_write.sum per launch, ncu --set full: profiles/{ent['source']}"
    except Exception:
        pass
    kname = (("fcnet_train_tc2_kernel" if K.tc_pingpong_eligible(D, A) else "fcnet_train_tc_kernel") +
             " (fused fwd + PPO loss + bwd + grad reduce + clip + Adam; tcgen05 kind::f16, fp16 hi/lo split x3 products, TMEM accum)"
             if args.mode == "tc" else "fcnet_train_kernel (fused fwd + PPO loss + bwd + grad reduce + clip + Adam, FP32 FMA parity mode)")
    roofline = {"bound": "tensor", "kernel": kname,
                "achieved": achieved_tf, "peak": tensor_peak, "unit": "TFLOP/s", "frac": achieved_tf / tensor_peak,
                "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained" if peaks else "fallback 1.4 PFLOP/s sustained",
                "traffic": traffic, "traffic_note": traffic_note,
                "launch_ms": k_ms, "flops_per_launch": flops_launch, "sgd_steps_per_launch": steps_per_launch,
                "us_per_sgd_step": 1e3 * k_ms / steps_per_launch,
                "note": "latency/issue-bound: 4096 rows x 4 policies per step = one 128-row tile per SM (DESIGN.md §4)",
                "share_of_step": (steps_per_iter / steps_per_launch) * k_ms / (ms_total / args.steps)}

    # replicated state must be bit-identical on every rank (SURVEY.md §8-e): 64-bit checksum of the weights and Adam slots
    def checksum(t):
        return t.contiguous().view(torch.int32).to(torch.int64).sum()
    cks = torch.stack([checksum(L.theta), checksum(L.m), checksum(L.v)])
    ranks_identical = True
    if world > 1:
        allc = [torch.empty_like(cks) for _ in range(world)]
        dist.all_gather(allc, cks)
        ranks_identical = all(bool(torch.equal(a_, allc[0])) for a_ in allc)
    supplementary = None
    if rank == 0 and world == 1 and not args.no_supplementary and args.arch == "FullyDecentral" and args.mode == "tc":
        supplementary = run_supplementary(args)

    line = None
    if rank == 0:
        cpu = None
        if not args.no_cpu_baseline and world == 1:      # rank 0 at N = 1 only (at N > 1 the other ranks would idle on metered GPUs)
            v, dt, threads = cpu_iteration_baseline(args.cpu_envs)
            cpu = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
                   "sample": f"{args.cpu_envs} of {envs} envs, one full learner iteration ({dt:.1f} s), torch CPU float32 twin of the oracle"}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if args.mode == "fp32" else "f32 (tcgen05 GEMMs on fp16 hi+lo split operands, f32 accumulate)",
            "data": "synthetic",
            "config": dict(workload_config(envs, world, nb, args.sets),
                           parallelism=(f"dp{world}: rollout sharded by env, one process per GPU; the gradient all-reduce of every optimizer "
                                        "step runs INSIDE the SGD-step kernel over NVLink peer memory (no NCCL call on the per-step "
                                        "path); NCCL only for the per-iteration filter / advantage-moment / stat exchanges")
                           if world > 1 else "single GPU"),
            "impl_detail": {"cuda_graph_prepare_phase": bool(L.use_graph and L._prep_graphs), "sgd_kernel": args.mode,
                            "kernels_per_sgd_step": per_sgd, "persistent_sgd_launch": bool(L._persistent_steps(G_)),
                            "ctas_per_policy": G_, "cluster_size": K.tc_last_cluster() if args.mode == "tc" else 0,
                            "partial_gradient_reduce": ("L2 accumulation vector (red.global.add.v4.f32; float addition order not fixed)"
                                                        if getattr(L, "atomic_reduce", False) and args.mode == "tc"
                                                        else "fixed-order sum of per-CTA partials"),
                            "bytes_per_rollout_set": int(bytes_per_set)},
            "ranks_identical": ranks_identical,
            "clocks": clk,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(nb * P * 8 * 8),
                    "inputs": "pinned host: full 43-dim observations per env step (+ boot obs, rewards, dones, perms, shuffle); "
                              "per-agent index gather on the device (ddrl_obs_gather); the copy of step i+1 overlaps the compute of step i "
                              "(double-buffered staging on a copy stream)",
                    "ms_per_step": ms_e2e / e2e_steps},
            "gpu_launches": int(launches_per_iter * args.steps),
            "api_launch_calls": int(K.launch_count() - n0),
            "roofline": roofline,
            "cpu_baseline": cpu,
            "flops_per_agent_step": flops_per_agent_step(D, A, E),
            "supplementary": supplementary,
        }
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(line), flush=True)
    if world > 1:
        # release the captured graph (it holds NCCL work) before tearing the communicator down, and never let the
        # teardown hang the job: the result line is already out
        L._graph = None
        torch.cuda.synchronize()
        dist.barrier()
        t = threading.Thread(target=dist.destroy_process_group, daemon=True)
        t.start()
        t.join(timeout=15.0)
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


if __name__ == "__main__":
    main()

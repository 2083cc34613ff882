"""Import / export of the reference's RLlib (Ray 1.0.x) PPO checkpoints without Ray or TensorFlow  (SURVEY.md §8-f N3).

File format (``Results/**/checkpoint_1250/checkpoint-1250``, written by ``Trainable.save`` of Ray 1.0.x; consumers:
``evaluation/evaluate_trained_policies_pd.py:84-96`` and ``show_trained_multiagent_policy.py:48-49`` through
``agent.restore``): two nested pickles ::

    top    = {"worker": <bytes>, "train_exec_impl": {"counters": {...}, "info": {"learner": {pid: stats}}, "timers": None}}
    worker = {"filters": {pid: MeanStdFilter(shape, demean, destd, clip, rs=RunningStat(_n, _M, _S), buffer=RunningStat)},
              "state":   {pid: OrderedDict["<pid>/fc_1/kernel" (D,64), "<pid>/fc_1/bias", "<pid>/fc_value_1/...",
                                           "<pid>/fc_2/...", "<pid>/fc_value_2/...", "<pid>/fc_out/..." (64,2A),
                                           "<pid>/value_out/..." (64,1),
                                           "_optimizer_variables": OrderedDict["<pid>/beta1_power", "<pid>/beta2_power",
                                               "<pid>/<var>/Adam" (m), "<pid>/<var>/Adam_1" (v), ...]]}}

The only non-numpy classes are ``ray.rllib.utils.filter.{MeanStdFilter, RunningStat}``; they are read through stub
classes and written under their real module path, so a file exported here restores in the reference's RLlib
(``agent.restore``) and a reference checkpoint continues training on ``FCNetLearner``.

The flat parameter order of this repo IS the checkpoint variable order (``FC_VARS``), so import / export are copies.
Pure host code (numpy + pickle); the learner side needs CUDA tensors only in ``apply_to_learner`` /
``from_learner``."""
from __future__ import annotations

import io
import pickle
import sys
import types
from collections import OrderedDict
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Tuple

import numpy as np

FC_VARS = ("fc_1", "fc_value_1", "fc_2", "fc_value_2", "fc_out", "value_out")
_FILTER_MODULE = "ray.rllib.utils.filter"


# ---- stub classes with the pickled attribute layout of ray.rllib.utils.filter -------------------------------------------
class RunningStat:
    """Attribute-compatible stand-in for ray.rllib.utils.filter.RunningStat (``_n`` int, ``_M`` / ``_S`` float64)."""

    def __init__(self, shape=()):
        self._n = 0
        self._M = np.zeros(shape, dtype=np.float64)
        self._S = np.zeros(shape, dtype=np.float64)

    def __setstate__(self, s):
        self.__dict__.update(s)


class MeanStdFilter:
    """Attribute-compatible stand-in for ray.rllib.utils.filter.MeanStdFilter."""

    def __init__(self, shape=(), demean=True, destd=True, clip=None):
        self.shape, self.demean, self.destd, self.clip = shape, demean, destd, clip
        self.rs = RunningStat(shape)
        self.buffer = RunningStat(shape)

    def __setstate__(self, s):
        self.__dict__.update(s)


class _StubUnpickler(pickle.Unpickler):
    def find_class(self, module, name):
        if module == _FILTER_MODULE and name in ("MeanStdFilter", "RunningStat"):
            return {"MeanStdFilter": MeanStdFilter, "RunningStat": RunningStat}[name]
        try:
            return super().find_class(module, name)
        except Exception:  # any other ray / tf class: keep its state as a plain attribute bag
            return type(name, (), {"__setstate__": lambda self, s: self.__dict__.update(s)})


# ---- in-memory form ------------------------------------------------------------------------------------------------------
@dataclass
class PolicyCheckpoint:
    """One policy of a checkpoint, in this repo's flat layout."""
    theta: np.ndarray                      # [NP] float32, checkpoint variable order
    shapes: List[Tuple[int, ...]]          # 12 variable shapes (kernel, bias) x FC_VARS
    adam_m: Optional[np.ndarray] = None    # [NP] float32 (TF1 slot "Adam")
    adam_v: Optional[np.ndarray] = None    # [NP] float32 (TF1 slot "Adam_1")
    beta_powers: Optional[np.ndarray] = None   # [2] float32 (beta1_power, beta2_power)
    filter_n: int = 0
    filter_M: Optional[np.ndarray] = None  # [D] float64
    filter_S: Optional[np.ndarray] = None  # [D] float64
    filter_clip: Optional[float] = None
    learner_stats: Dict[str, float] = field(default_factory=dict)   # incl. cur_kl_coeff, cur_lr

    @property
    def obs_dim(self) -> int:
        return int(self.shapes[0][0])

    @property
    def act_dim(self) -> int:
        return int(self.shapes[8][1]) // 2


@dataclass
class Checkpoint:
    policies: "OrderedDict[str, PolicyCheckpoint]"
    counters: Dict[str, int] = field(default_factory=dict)


def _flatten(pid: str, src, suffix: str = ""):
    chunks, shapes = [], []
    for layer in FC_VARS:
        for part in ("kernel", "bias"):
            key = f"{pid}/{layer}/{part}"
            if suffix:
                key = f"{pid}/{key}{suffix}"
            a = np.asarray(src[key], dtype=np.float32)
            shapes.append(tuple(a.shape))
            chunks.append(a.reshape(-1))
    return np.concatenate(chunks), shapes


def load_rllib_checkpoint(path: str) -> Checkpoint:
    """Read a ``checkpoint-N`` file of the reference (Ray 1.0.x PPO, FCNet policies)."""
    with open(path, "rb") as f:
        top = _StubUnpickler(f).load()
    worker = _StubUnpickler(io.BytesIO(top["worker"])).load()
    stats = (top.get("train_exec_impl") or {}).get("info", {}).get("learner", {})
    pols: "OrderedDict[str, PolicyCheckpoint]" = OrderedDict()
    for pid, od in worker["state"].items():
        theta, shapes = _flatten(pid, od)
        pc = PolicyCheckpoint(theta=theta, shapes=shapes)
        opt = od.get("_optimizer_variables")
        if opt:
            pc.adam_m, _ = _flatten(pid, opt, "/Adam")
            pc.adam_v, _ = _flatten(pid, opt, "/Adam_1")
            pc.beta_powers = np.asarray([opt[f"{pid}/beta1_power"], opt[f"{pid}/beta2_power"]], dtype=np.float32)
        flt = worker.get("filters", {}).get(pid)
        if flt is not None and hasattr(flt, "rs"):
            pc.filter_n = int(flt.rs._n)
            pc.filter_M = np.asarray(flt.rs._M, dtype=np.float64).reshape(-1).copy()
            pc.filter_S = np.asarray(flt.rs._S, dtype=np.float64).reshape(-1).copy()
            pc.filter_clip = getattr(flt, "clip", None)
        pc.learner_stats = {k: float(v) for k, v in stats.get(pid, {}).items() if np.isscalar(v) or isinstance(v, np.generic)}
        pols[pid] = pc
    counters = dict((top.get("train_exec_impl") or {}).get("counters", {}) or {})
    return Checkpoint(policies=pols, counters=counters)


def _unflatten(pid: str, flat: np.ndarray, shapes, suffix: str = "", prefix_pid: bool = False) -> "OrderedDict[str, np.ndarray]":
    out: "OrderedDict[str, np.ndarray]" = OrderedDict()
    o, i = 0, 0
    for layer in FC_VARS:
        for part in ("kernel", "bias"):
            shp = tuple(int(s) for s in shapes[i])
            n = int(np.prod(shp))
            key = f"{pid}/{layer}/{part}"
            if prefix_pid:
                key = f"{pid}/{key}{suffix}"
            out[key] = np.asarray(flat[o:o + n], dtype=np.float32).reshape(shp).copy()
            o += n
            i += 1
    if o != flat.size:
        raise ValueError(f"flat vector has {flat.size} entries, the variable shapes need {o}")
    return out


def fcnet_variable_shapes(D: int, A: int) -> List[tuple]:
    """Shapes of the 12 FCNet variables in checkpoint order (hiddens [64, 64], separate value branch)."""
    return [(D, 64), (64,), (D, 64), (64,), (64, 64), (64,), (64, 64), (64,), (64, 2 * A), (2 * A,), (64, 1), (1,)]


def theta_to_variables(pid: str, theta: np.ndarray, D: int, A: int) -> "OrderedDict[str, np.ndarray]":
    """Flat parameter vector -> {"<pid>/fc_1/kernel": ..., ...}: what `Policy.get_weights()` returns in the reference."""
    return _unflatten(pid, np.asarray(theta, dtype=np.float32).reshape(-1), fcnet_variable_shapes(D, A))


def variables_to_theta(pid: str, variables, D: int, A: int) -> np.ndarray:
    """Inverse of `theta_to_variables` (`Policy.set_weights`); shapes are checked against the (D, A) architecture."""
    theta, shapes = _flatten(pid, variables)
    if [tuple(s) for s in shapes] != fcnet_variable_shapes(D, A):
        raise ValueError(f"{pid}: variable shapes {shapes} do not match FCNet(D={D}, A={A})")
    return theta


def save_rllib_checkpoint(path: str, ckpt: Checkpoint) -> None:
    """Write ``ckpt`` in the reference's file format (see module docstring).  The filter classes are pickled under
    ``ray.rllib.utils.filter`` so that the reference's ``agent.restore`` resolves them to the real RLlib classes."""
    state, filters, learner = OrderedDict(), {}, {}
    for pid, pc in ckpt.policies.items():
        od = _unflatten(pid, pc.theta, pc.shapes)
        if pc.adam_m is not None and pc.adam_v is not None:
            opt: "OrderedDict[str, np.ndarray]" = OrderedDict()
            bp = pc.beta_powers if pc.beta_powers is not None else np.asarray([0.9, 0.999], np.float32)
            opt[f"{pid}/beta1_power"] = np.float32(bp[0])
            opt[f"{pid}/beta2_power"] = np.float32(bp[1])
            m = _unflatten(pid, pc.adam_m, pc.shapes, "/Adam", True)
            v = _unflatten(pid, pc.adam_v, pc.shapes, "/Adam_1", True)
            for (km, am), (kv, av) in zip(m.items(), v.items()):   # TF order: var/Adam, var/Adam_1, next var ...
                opt[km] = am
                opt[kv] = av
            od["_optimizer_variables"] = opt
        state[pid] = od
        if pc.filter_M is not None:
            f = MeanStdFilter(tuple(pc.filter_M.shape), True, True, pc.filter_clip)
            f.rs._n = int(pc.filter_n)
            f.rs._M = np.asarray(pc.filter_M, np.float64).copy()
            f.rs._S = np.asarray(pc.filter_S, np.float64).copy()
            filters[pid] = f
        st = dict(pc.learner_stats)
        learner[pid] = {k: (np.float64(v) if k in ("cur_kl_coeff", "cur_lr", "entropy_coeff") else np.float32(v)) for k, v in st.items()}
        learner[pid]["model"] = {}
    # pickle resolves classes by module path at dump time: provide ray.rllib.utils.filter for the duration of the dump
    created = []
    parts = _FILTER_MODULE.split(".")
    for i in range(1, len(parts) + 1):
        name = ".".join(parts[:i])
        if name not in sys.modules:
            sys.modules[name] = types.ModuleType(name)
            created.append(name)
    mod = sys.modules[_FILTER_MODULE]
    saved = {n: getattr(mod, n, None) for n in ("MeanStdFilter", "RunningStat")}
    old_meta = {c: (c.__module__, c.__qualname__) for c in (MeanStdFilter, RunningStat)}
    try:
        for c in (MeanStdFilter, RunningStat):
            setattr(mod, c.__name__, c)
            c.__module__ = _FILTER_MODULE
        worker = pickle.dumps({"filters": filters, "state": state}, protocol=4)
        top = {"worker": worker,
               "train_exec_impl": {"counters": dict(ckpt.counters), "info": {"learner": learner}, "timers": None}}
        with open(path, "wb") as f:
            pickle.dump(top, f, protocol=4)
    finally:
        for c, (m, q) in old_meta.items():
            c.__module__ = m
        for n, v in saved.items():
            if v is None:
                if hasattr(mod, n):
                    delattr(mod, n)
            else:
                setattr(mod, n, v)
        for name in reversed(created):
            sys.modules.pop(name, None)


# ---- learner <-> checkpoint ---------------------------------------------------------------------------------------------
def _reject_coupled(learner) -> None:
    from .learner import GraphNetLearner
    if isinstance(learner, GraphNetLearner):
        raise ValueError("checkpoints of the shared GraphNet policy are not supported: no GraphNet checkpoint was published, "
                         "so none pins the format; use GraphNetPolicyGroup.get_weights / set_weights")
    if getattr(learner, "coupled", False):
        raise ValueError("checkpoints of leg-coupled ('cup') policies are not supported: no reference checkpoint pins the "
                         "naming of the leg_coupling variable; use get_weights / set_weights")


def apply_to_learner(ckpt: Checkpoint, learner, policy_ids: Optional[List[str]] = None) -> None:
    """Load weights, Adam moments / beta powers, filter state and KL coefficients into an ``FCNetLearner`` (policy slot
    p <- policy_ids[p], default: checkpoint order)."""
    import torch
    _reject_coupled(learner)
    pids = list(policy_ids or ckpt.policies.keys())
    if len(pids) != learner.P:
        raise ValueError(f"checkpoint has {len(pids)} policies, learner {learner.P}")
    dev = learner.device
    for p, pid in enumerate(pids):
        pc = ckpt.policies[pid]
        if pc.theta.size != learner.NP or pc.obs_dim != learner.D or pc.act_dim != learner.A:
            raise ValueError(f"policy {pid}: checkpoint (D={pc.obs_dim}, A={pc.act_dim}, NP={pc.theta.size}) does not match "
                             f"the learner (D={learner.D}, A={learner.A}, NP={learner.NP})")
        learner.theta[p].copy_(torch.from_numpy(pc.theta).to(dev))
        if pc.adam_m is not None:
            learner.m[p].copy_(torch.from_numpy(pc.adam_m).to(dev))
            learner.v[p].copy_(torch.from_numpy(pc.adam_v).to(dev))
        if pc.beta_powers is not None:
            learner.beta_pow[p].copy_(torch.from_numpy(np.asarray(pc.beta_powers, np.float32)).to(dev))
        if pc.filter_M is not None:
            learner.filt_n[p] = int(pc.filter_n)
            learner.filt_M[p].copy_(torch.from_numpy(pc.filter_M).to(dev))
            learner.filt_S[p].copy_(torch.from_numpy(pc.filter_S).to(dev))
        if "cur_kl_coeff" in pc.learner_stats:
            learner.kl_coeff_host[p] = float(pc.learner_stats["cur_kl_coeff"])
    learner.kl_coeff.copy_(torch.from_numpy(learner.kl_coeff_host.astype(np.float32)).to(dev))
    learner.refresh_filter_norm()


def from_learner(learner, policy_ids: List[str], stats: Optional[List[Dict[str, float]]] = None,
                 counters: Optional[Dict[str, int]] = None) -> Checkpoint:
    """Snapshot an ``FCNetLearner`` as a ``Checkpoint`` (``stats`` = the list ``learn_on_rollout`` returned)."""
    _reject_coupled(learner)
    D, A = learner.D, learner.A
    shapes = [(D, 64), (64,), (D, 64), (64,), (64, 64), (64,), (64, 64), (64,), (64, 2 * A), (2 * A,), (64, 1), (1,)]
    pols: "OrderedDict[str, PolicyCheckpoint]" = OrderedDict()
    for p, pid in enumerate(policy_ids):
        st = dict(stats[p]) if stats else {}
        # the coefficient the NEXT iteration will use (RLlib's own stat is the pre-update value and its checkpoints do not
        # carry the kl_coeff variable at all — a restored RLlib trainer restarts from config["kl_coeff"])
        st["cur_kl_coeff"] = float(learner.kl_coeff_host[p])
        st.setdefault("cur_lr", float(np.float32(learner.cfg.lr)))
        pols[pid] = PolicyCheckpoint(
            theta=learner.theta[p].detach().cpu().numpy().copy(), shapes=shapes,
            adam_m=learner.m[p].cpu().numpy().copy(), adam_v=learner.v[p].cpu().numpy().copy(),
            beta_powers=learner.beta_pow[p].cpu().numpy().copy(),
            filter_n=int(learner.filt_n[p].item()), filter_M=learner.filt_M[p].cpu().numpy().copy(),
            filter_S=learner.filt_S[p].cpu().numpy().copy(), filter_clip=learner.cfg.filter_clip, learner_stats=st)
    return Checkpoint(policies=pols, counters=dict(counters or {}))

"""RLlib-facing learner surface (SURVEY.md §8-f N4): the calls RLlib 1.0.1 makes on a PPO policy, served by the fused
B200 learner for ALL policies of an architecture at once.

RLlib's execution plan (`ray/rllib/agents/ppo/ppo.py` `execution_plan`, driven by the reference through
`tune.run("PPO", config=...)`, train_experiment_1_architecture_on_flat.py:201-211) does, per training iteration:

    rollout workers: obs -> MeanStdFilter -> Policy.compute_actions -> SampleBatch rows
                     Policy.postprocess_trajectory (postprocess_ppo_gae) per episode fragment
    driver:          ConcatBatches -> StandardizeFields(["advantages"]) -> TrainTFMultiGPU / TrainOneStep:
                     for every policy id in the MultiAgentBatch: Policy.learn_on_batch(batch)   (1250 session.run each)
                     UpdateKL

`PPOPolicyGroup` mirrors that surface with the reference's column names (`SampleBatch.OBS` = "obs", "actions",
"action_dist_inputs", "action_logp", "vf_preds", "advantages", "value_targets", "rewards", "dones", "new_obs"):
`compute_actions`, `postprocess_fragments` (batched `postprocess_ppo_gae`), `learn_on_batch` (a MultiAgentBatch-like
`{policy_id: {column: array}}` in, `{policy_id: {"learner_stats": {...}}}` out — the shape `RolloutWorker.learn_on_batch`
returns), `get_weights` / `set_weights` with the TF variable names of the reference checkpoints, and
`update_environment_after_epoch` for the `on_train_result` curriculum callback
(train_experiment_1_architecture_on_flat.py:171-178).  With ray installed the train op of a custom execution plan calls
`learn_on_batch` on the concatenated MultiAgentBatch; ray is absent in this image, so that glue is shown in
INTEGRATION.md §4.1, not shipped.

`GraphNetPolicyGroup` serves the shared GraphNet policy of QuantrupedMultiEnv_DecentralShared_Graph (model "gnn") with
the same calls, over the Tuple observation (node_idx, state, adj).

Everything that computes runs on the GPU through `learner.FCNetLearner` / `learner.GraphNetLearner` / the C ABI; this
module only validates and stacks host arrays, draws the permutations RLlib would draw (numpy RandomState) and copies to /
from the device."""
from __future__ import annotations

from typing import Any, Dict, List, Mapping, Optional, Sequence, Tuple

import numpy as np

from . import policies as _policies
from .config import PPOConfig

OBS, NEXT_OBS, ACTIONS, REWARDS, DONES = "obs", "new_obs", "actions", "rewards", "dones"
ACTION_DIST_INPUTS, ACTION_LOGP, VF_PREDS = "action_dist_inputs", "action_logp", "vf_preds"
ADVANTAGES, VALUE_TARGETS = "advantages", "value_targets"
TRAIN_COLUMNS = (OBS, ACTIONS, ACTION_DIST_INPUTS, ACTION_LOGP, VF_PREDS, ADVANTAGES, VALUE_TARGETS)


NODE_IDX = "node_idx"      # leg-coupled / graph policies: the Discrete(4) node-id part of the Tuple observation
ADJ = "adj"                # graph policy: the MultiDiscrete(2) [4, 4] adjacency part of the Tuple observation
GRAPH_NODES, GRAPH_NODE_WIDTH = 4, 23      # shared GraphNet state [4, 19 + 4]


class BatchError(ValueError):
    pass


def check_node_idx(node_idx, rows: int, where: str) -> np.ndarray:
    """The node-id part of the SharedDecentralLegID observation: [rows] integers 0..3 (FL, HL, HR, FR) -> int32."""
    a = np.asarray(node_idx)
    if a.ndim == 2 and a.shape[1] == 1:
        a = a[:, 0]
    if a.ndim != 1 or a.shape[0] != rows:
        raise BatchError(f"{where}: node_idx must have shape [{rows}], got {a.shape}")
    if a.dtype.kind not in "iu" and not (a.dtype.kind == "f" and np.all(np.isfinite(a)) and np.all(a == np.round(a))):
        raise BatchError(f"{where}: node_idx must hold integers, got {a.dtype}")
    if a.size and (a.min() < 0 or a.max() > 3):
        raise BatchError(f"{where}: node_idx must be in 0..3 (FL, HL, HR, FR), got range [{a.min()}, {a.max()}]")
    return np.ascontiguousarray(a.astype(np.int32))


def check_graph_obs(node_idx, state, adj, where: str) -> Tuple[np.ndarray, np.ndarray, np.ndarray]:
    """The Tuple observation of the shared GraphNet policy: node_idx [B] (or [B, 1]) integers 0..3, state [B, 4, 23] finite
    floats, adj [B, 4, 4] with entries in {0, 1} (the MultiDiscrete(2) space) -> int32 [B], float32 [B, 4, 23], float32
    [B, 4, 4]."""
    st = np.asarray(state)
    if st.ndim != 3 or st.shape[1:] != (GRAPH_NODES, GRAPH_NODE_WIDTH) or st.dtype.kind != "f":
        raise BatchError(f"{where}: state must be a float array of shape [B, {GRAPH_NODES}, {GRAPH_NODE_WIDTH}], "
                         f"got {st.dtype} {st.shape}")
    with np.errstate(over="ignore"):      # float64 beyond the float32 range becomes inf and is rejected below
        st = np.ascontiguousarray(st, dtype=np.float32)
    if not np.isfinite(st).all():
        raise BatchError(f"{where}: state contains non-finite values")
    B = st.shape[0]
    node = check_node_idx(node_idx, B, where)
    a = np.asarray(adj)
    if a.shape != (B, GRAPH_NODES, GRAPH_NODES):
        raise BatchError(f"{where}: adj must have shape [{B}, {GRAPH_NODES}, {GRAPH_NODES}], got {a.shape}")
    if not np.isin(a, (0, 1)).all():
        raise BatchError(f"{where}: adj entries must be 0 or 1 (MultiDiscrete(2) space)")
    return node, st, np.ascontiguousarray(a, dtype=np.float32)


def stack_policy_batches(policy_batches: Mapping[str, Mapping[str, Any]], policy_names: Sequence[str], D: int, A: int,
                         columns: Sequence[str] = TRAIN_COLUMNS) -> Dict[str, np.ndarray]:
    """{policy_id: {column: [R, ...]}} -> {column: float32 [P, R, ...]} in `policy_names` order.

    The fused learner trains the P policies of an architecture in ONE launch, so their batches must have the same
    number of rows — which the reference's environments guarantee (every agent acts at every env step,
    quantruped_adaptor_multi_environment.py:214-246).  Missing policies / columns, ragged row counts, wrong widths and
    non-finite values are errors (RLlib would feed them to TF and train on them)."""
    missing = [p for p in policy_names if p not in policy_batches]
    if missing:
        raise BatchError(f"policy_batches lacks {missing}; policies_to_train = {list(policy_names)}")
    extra = [p for p in policy_batches if p not in policy_names]
    if extra:
        raise BatchError(f"unknown policy ids {extra}; this group trains {list(policy_names)}")
    width = {OBS: D, NEXT_OBS: D, ACTIONS: A, ACTION_DIST_INPUTS: 2 * A}
    out: Dict[str, np.ndarray] = {}
    rows: Optional[int] = None
    for col in columns:
        per_policy = []
        for p in policy_names:
            if col not in policy_batches[p]:
                raise BatchError(f"batch of {p!r} lacks column {col!r}")
            a = np.asarray(policy_batches[p][col])
            want_nd = 2 if col in width else 1
            if a.ndim != want_nd or (col in width and a.shape[1] != width[col]):
                raise BatchError(f"{p}/{col}: expected shape [R{', %d' % width[col] if col in width else ''}], got {a.shape}")
            if rows is None:
                rows = a.shape[0]
            if a.shape[0] != rows:
                raise BatchError(f"{p}/{col} has {a.shape[0]} rows, other columns have {rows}: the grouped learner needs "
                                 "equally long batches for all policies")
            a = a.astype(np.float32, copy=False)
            if not np.isfinite(a).all():
                raise BatchError(f"{p}/{col} contains non-finite values")
            per_policy.append(a)
        out[col] = np.ascontiguousarray(np.stack(per_policy))
    if not rows:
        raise BatchError("empty train batch")
    return out


def draw_minibatch_order(rng: np.random.RandomState, P: int, R: int, num_sgd_iter: int, minibatches: int,
                         shuffle_sequences: bool = True) -> Tuple[Optional[np.ndarray], np.ndarray]:
    """The random draws of RLlib's multi-GPU optimizer, per policy in policy order: one `SampleBatch.shuffle()`
    (`np.random.permutation(R)`, only with `shuffle_sequences`) and one `np.random.permutation(num_batches)` per SGD
    epoch (`TrainTFMultiGPU`, ray/rllib/execution/train_ops.py).  -> shuffle [P, R] int32 | None, perms [P, E, nb] int32."""
    shuffle = None
    if shuffle_sequences:
        shuffle = np.stack([rng.permutation(R) for _ in range(P)]).astype(np.int32)
    perms = np.stack([np.stack([rng.permutation(minibatches) for _ in range(num_sgd_iter)]) for _ in range(P)])
    return shuffle, perms.astype(np.int32)


def usable_rows(R: int, sgd_minibatch_size: int) -> Tuple[int, int]:
    """RLlib's multi-GPU loader truncates the batch to a whole number of minibatches: (rows used, minibatches)."""
    mb = min(int(sgd_minibatch_size), R)
    nb = R // mb
    return nb * mb, nb


def curriculum_smoothness(timesteps_total: float, initial: float, target: float, last_timestep: float, u: float) -> float:
    """Height-field smoothness after a training iteration (`update_environment_after_epoch`,
    quantruped_adaptor_multi_environment.py:97-122), `u` = the `np.random.rand()` draw: inside the curriculum interval a
    random point between flat and the linearly decreasing bound, afterwards anywhere between target and flat."""
    if last_timestep > timesteps_total:
        return initial - u * (initial - target) * (timesteps_total / last_timestep)
    return target + u * (initial - target)


class _PolicyGroupBase:
    """What every policy group shares: the RLlib config, the group's RandomState (action noise, minibatch order, curriculum
    draws), the GAE postprocessing, RLlib's batch preparation order and the curriculum callback.  Subclasses set
    `self.learner` (with `standardize_advantages`)."""

    def _init_common(self, config: Optional[Dict[str, Any]], device, seed: Optional[int]) -> None:
        import torch
        self.config = dict(config or {})
        self.ppo = PPOConfig.from_rllib(self.config)
        self.device = torch.device(device)
        self.rng = np.random.RandomState(self.config.get("seed", seed))
        self.shuffle_sequences = bool(self.config.get("shuffle_sequences", True))
        self.num_steps_trained = 0
        self.current_smoothness: Optional[float] = None

    def postprocess_fragments(self, rewards: np.ndarray, vf_preds: np.ndarray, dones: np.ndarray, last_values: np.ndarray):
        """Batched `postprocess_ppo_gae` (RLlib evaluation/postprocessing.py): rewards / vf_preds [P, T, C] for C
        fragment columns of T steps, dones [T, C] (episode ended AT that step), last_values [P, C] = V(new_obs[-1]) of
        each column (ignored where the column's last step is done) -> (advantages, value_targets) [P, T, C]."""
        import torch
        from . import kernels as K
        to = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).to(self.device)
        adv, vtarg, _ = K.gae(to(rewards, np.float32), to(vf_preds, np.float32), to(dones, np.uint8), to(last_values, np.float32),
                              1, self.ppo.gamma, self.ppo.lambda_)
        return adv.cpu().numpy(), vtarg.cpu().numpy()

    def _prepare_batch(self, d: Dict[str, Any], R: int, standardize: bool):
        """RLlib's order on a train batch d = {column: [P, R, ...] device tensor}: the RandomState draws (shuffle, then the
        per-epoch minibatch permutations), StandardizeFields over ALL R rows, then the multi-GPU loader's truncation to whole
        minibatches (the first `used` rows of the shuffled batch; no shuffle is passed on after it).
        -> (d, shuffle [P, R] or None, perms [P, E, nb], used)."""
        import torch
        P = d[ADVANTAGES].shape[0]
        used, nb = usable_rows(R, self.ppo.sgd_minibatch_size)
        shuffle, perms = draw_minibatch_order(self.rng, P, R, self.ppo.num_sgd_iter, nb, self.shuffle_sequences)
        dev = lambda a: torch.from_numpy(a).to(self.device)
        if standardize:        # StandardizeFields sees the WHOLE train batch, before the loader drops the ragged tail
            self.learner.standardize_advantages(d[ADVANTAGES])
        shuf = None if shuffle is None else dev(shuffle)
        if used != R:          # the multi-GPU loader keeps whole minibatches: the first `used` rows of the shuffled batch
            keep = (shuf[:, :used] if shuf is not None else torch.arange(used, device=self.device).expand(P, used)).long()
            d = {k: torch.gather(v, 1, keep.reshape(P, used, *([1] * (v.dim() - 2))).expand(P, used, *v.shape[2:])).contiguous()
                 for k, v in d.items()}
            shuf = None
        return d, shuf, dev(perms), used

    def update_environment_after_epoch(self, timesteps_total: float) -> Optional[float]:
        """What `on_train_result` makes every env do (train_experiment_1_architecture_on_flat.py:171-178): returns the new
        height-field smoothness for the simulator (None when `curriculum_learning` is off)."""
        ec = self.config.get("env_config", {})
        if not ec.get("curriculum_learning", False):
            return None
        lo, hi = ec["range_smoothness"]
        self.current_smoothness = curriculum_smoothness(timesteps_total, lo, hi, ec["range_last_timestep"], self.rng.rand())
        return self.current_smoothness


class PPOPolicyGroup(_PolicyGroupBase):
    """All policies of one `--policy_scope` behind one fused learner; see the module docstring.  `learner_kw` goes to
    `FCNetLearner`, among them filter_mode / filter_workers: with filter_mode="stream" every
    `compute_actions(update_filter=True)` call filters its rows one by one, as the sampler of an RLlib rollout worker calls
    the policy's MeanStdFilter once per observation — the mode an RLlib drop-in should use; the default "batch" is the
    vectorised filter call (all rows pushed, then all normalised with the final statistics)."""

    def __init__(self, policy_scope: str, config: Optional[Dict[str, Any]] = None, device="cuda", seed: Optional[int] = None,
                 use_target_velocity: bool = False, **learner_kw):
        from .learner import FCNetLearner
        env = _policies.ARCHITECTURES[policy_scope]
        self.coupled = getattr(env, "model", "fc_glorot_uniform_init") == "cup"
        if self.coupled:
            learner_kw = dict(learner_kw, leg_coupling=True)
        elif getattr(env, "model", "fc_glorot_uniform_init") != "fc_glorot_uniform_init":
            raise NotImplementedError(f"{policy_scope}: PPOPolicyGroup serves the FCNet architectures; the shared GraphNet "
                                      "policy is served by GraphNetPolicyGroup")
        self.env = env
        self.policy_names: List[str] = list(env.policy_names)
        self._init_common(config, device, seed)
        self.D, self.A = env.obs_dim(use_target_velocity), env.act_dim()
        self.learner = FCNetLearner(len(self.policy_names), self.D, self.A, self.ppo, self.device, **learner_kw)

    # ---- sampler side -------------------------------------------------------------------------------------------------
    def compute_actions(self, obs_by_policy: Mapping[str, np.ndarray], explore: bool = True, update_filter: bool = False):
        """`Policy.compute_actions` for every policy at once: {pid: raw obs [B, D]} ->
        {pid: (actions [B, A], [], {"action_dist_inputs", "action_logp", "vf_preds"})}.  With `explore` actions are
        DiagGaussian samples (noise from this group's RandomState), otherwise the distribution mean (logp of the mean).
        Leg-coupled policy (SharedDecentralLegID): {pid: (node_idx [B], obs [B, D])} — the Tuple observation."""
        import torch
        node = None
        if self.coupled:
            pid = self.policy_names[0]
            if set(obs_by_policy) != {pid}:
                raise BatchError(f"expected observations of {pid!r} only, got {list(obs_by_policy)}")
            tup = obs_by_policy[pid]
            if not isinstance(tup, (tuple, list)) or len(tup) != 2:
                raise BatchError(f"{pid}: the observation is the tuple (node_idx [B], obs [B, D])")
            node_h = check_node_idx(tup[0], np.asarray(tup[1]).shape[0], pid)
            node = torch.from_numpy(node_h[None]).to(self.device)
            obs_by_policy = {pid: tup[1]}
        obs = stack_policy_batches({p: {OBS: obs_by_policy[p]} for p in obs_by_policy}, self.policy_names, self.D, self.A, (OBS,))[OBS]
        P, B = obs.shape[:2]
        noise = self.rng.standard_normal((P, B, self.A)).astype(np.float32) if explore else np.zeros((P, B, self.A), np.float32)
        out = self.learner.compute_actions(torch.from_numpy(obs).to(self.device), torch.from_numpy(noise).to(self.device),
                                           update_filter=update_filter, **({"node_idx": node} if self.coupled else {}))
        host = {k: v.cpu().numpy() for k, v in out.items() if v is not None}
        res = {}
        for i, p in enumerate(self.policy_names):
            info = {ACTION_DIST_INPUTS: host["logits"][i], ACTION_LOGP: host["logp"][i], VF_PREDS: host["value"][i]}
            res[p] = (host["action"][i], [], info)
        return res

    # ---- learner side -------------------------------------------------------------------------------------------------
    def learn_on_batch(self, policy_batches: Mapping[str, Mapping[str, Any]], standardize: bool = True):
        """`RolloutWorker.learn_on_batch(MultiAgentBatch)`: one PPO update of every policy from postprocessed columns."""
        import torch
        node = None
        if self.coupled:      # the node-id column beside the Box part of the observation
            pid = self.policy_names[0]
            pb = policy_batches.get(pid, {})
            if NODE_IDX not in pb:
                raise BatchError(f"batch of {pid!r} lacks column {NODE_IDX!r} (the node-id part of the observation)")
            node = check_node_idx(pb[NODE_IDX], np.asarray(pb[OBS]).shape[0], f"{pid}/{NODE_IDX}")[None]
            policy_batches = {p: {k: v for k, v in b.items() if k != NODE_IDX} for p, b in policy_batches.items()}
        cols = stack_policy_batches(policy_batches, self.policy_names, self.D, self.A)
        R = cols[OBS].shape[1]
        dev = lambda a: torch.from_numpy(a).to(self.device)
        d = {k: dev(v) for k, v in cols.items()}
        if node is not None:
            d[NODE_IDX] = dev(node)
        d, shuf, perms, used = self._prepare_batch(d, R, standardize)
        stats = self.learner.learn_on_batch(d[OBS], d[ACTIONS], d[ACTION_DIST_INPUTS], d[ACTION_LOGP], d[VF_PREDS],
                                            d[ADVANTAGES], d[VALUE_TARGETS], perms, shuf, standardize=False,
                                            node_idx=d.get(NODE_IDX))
        self.num_steps_trained += used
        return {p: {"learner_stats": stats[i]} for i, p in enumerate(self.policy_names)}

    # ---- weights (TF variable names of the reference checkpoints) -----------------------------------------------------
    def get_weights(self) -> Dict[str, Dict[str, np.ndarray]]:
        from .checkpoint import theta_to_variables
        th = self.learner.theta.cpu().numpy()
        NPf = self.learner.NPf
        out = {p: theta_to_variables(p, th[i, :NPf], self.D, self.A) for i, p in enumerate(self.policy_names)}
        if self.coupled:      # the registration order of the ModelV2 class: the 12 FCNet variables, then the table
            for i, p in enumerate(self.policy_names):
                out[p][f"{p}/leg_coupling"] = th[i, NPf:].reshape(4, 2).copy()
        return out

    def set_weights(self, weights: Mapping[str, Mapping[str, np.ndarray]]) -> None:
        import torch
        from .checkpoint import variables_to_theta
        th = np.stack([variables_to_theta(p, weights[p], self.D, self.A) for p in self.policy_names]).astype(np.float32)
        if self.coupled:
            tabs = []
            for p in self.policy_names:
                t = np.asarray(weights[p].get(f"{p}/leg_coupling"), dtype=np.float32) if f"{p}/leg_coupling" in weights[p] else None
                if t is None or t.shape != (4, 2):
                    raise ValueError(f"{p}: set_weights needs '{p}/leg_coupling' of shape (4, 2)")
                tabs.append(t.reshape(-1))
            th = np.concatenate([th, np.stack(tabs)], axis=1)
        self.learner.theta.copy_(torch.from_numpy(th).to(self.device))


class GraphNetPolicyGroup(_PolicyGroupBase):
    """The shared GraphNet policy of QuantrupedMultiEnv_DecentralShared_Graph (model "gnn": actor GraphNet(2A) + critic
    GraphNet(1), models/shared_graphnet_glorot_uniform_init.py) behind one `learner.GraphNetLearner`, with the method names
    and return shapes of `PPOPolicyGroup`.  The observation is the Tuple (node_idx [B], state [B, 4, 23], adj [B, 4, 4]);
    the graph env normalises it itself, so there is no filter argument.  `learner_kw` goes to `GraphNetLearner`
    (step="tc" | "three-kernel")."""

    def __init__(self, policy_scope: str = "QuantrupedMultiEnv_DecentralShared_Graph", config: Optional[Dict[str, Any]] = None,
                 device="cuda", seed: Optional[int] = None, use_target_velocity: bool = False, **learner_kw):
        from .learner import GraphNetLearner
        env = _policies.ARCHITECTURES[policy_scope]
        if getattr(env, "model", "fc_glorot_uniform_init") != "gnn":
            raise ValueError(f"{policy_scope}: GraphNetPolicyGroup serves the shared GraphNet policy; this scope is served by "
                             "PPOPolicyGroup")
        if env is not _policies.QuantrupedDecentralizedSharedGraphEnv:
            raise NotImplementedError(f"{policy_scope}: its node width 19 has no leg-encoding columns and does not fit "
                                      "GraphNet's state[..., -4:] split; only QuantrupedMultiEnv_DecentralShared_Graph is served")
        if use_target_velocity:
            raise NotImplementedError("GraphNetPolicyGroup: use_target_velocity is not supported — the reference GraphNet "
                                      "hard-codes the leg-feature width 19 (models/graph_net.py), so the target-velocity "
                                      "column does not fit")
        self.env = env
        self.policy_names: List[str] = list(env.policy_names)
        self._init_common(config, device, seed)
        self.A = env.act_dim()
        self.learner = GraphNetLearner(self.A, self.ppo, self.device, **learner_kw)

    def _tuple_obs(self, obs_by_policy: Mapping[str, Any]):
        pid = self.policy_names[0]
        if set(obs_by_policy) != {pid}:
            raise BatchError(f"expected observations of {pid!r} only, got {list(obs_by_policy)}")
        tup = obs_by_policy[pid]
        if not isinstance(tup, (tuple, list)) or len(tup) != 3:
            raise BatchError(f"{pid}: the observation is the tuple (node_idx [B], state [B, 4, 23], adj [B, 4, 4])")
        return check_graph_obs(tup[0], tup[1], tup[2], pid)

    # ---- sampler side -------------------------------------------------------------------------------------------------
    def compute_actions(self, obs_by_policy: Mapping[str, Any], explore: bool = True):
        """`Policy.compute_actions`: {pid: (node_idx [B], state [B, 4, 23], adj [B, 4, 4])} ->
        {pid: (actions [B, A], [], {"action_dist_inputs", "action_logp", "vf_preds"})}, in ONE kernel launch
        (`ddrl_graphnet_act`).  With `explore` the actions are DiagGaussian samples (noise from this group's RandomState,
        drawn as `standard_normal((1, B, A))` like `PPOPolicyGroup`), otherwise the distribution mean (logp of the mean)."""
        import torch
        node, state, adj = self._tuple_obs(obs_by_policy)
        B = state.shape[0]
        noise = self.rng.standard_normal((1, B, self.A)).astype(np.float32) if explore else np.zeros((1, B, self.A), np.float32)
        dev = lambda a: torch.from_numpy(a).to(self.device)
        out = self.learner.compute_actions(dev(node), dev(state), dev(adj), dev(noise[0]))
        host = {k: v.cpu().numpy() for k, v in out.items()}
        info = {ACTION_DIST_INPUTS: host["logits"], ACTION_LOGP: host["logp"], VF_PREDS: host["value"]}
        return {self.policy_names[0]: (host["action"], [], info)}

    # ---- learner side -------------------------------------------------------------------------------------------------
    def learn_on_batch(self, policy_batches: Mapping[str, Mapping[str, Any]], standardize: bool = True):
        """`RolloutWorker.learn_on_batch`: one PPO update from postprocessed columns {pid: {"node_idx" [R], "obs" = state
        [R, 4, 23], "adj" [R, 4, 4], "actions", "action_dist_inputs", "action_logp", "vf_preds", "advantages",
        "value_targets"}}, in `PPOPolicyGroup.learn_on_batch`'s order: RandomState draws, StandardizeFields over all R rows,
        truncation to whole minibatches, then `GraphNetLearner.learn_on_batch`."""
        import torch
        pid = self.policy_names[0]
        if set(policy_batches) != {pid}:
            raise BatchError(f"expected the batch of {pid!r} only, got {list(policy_batches)}")
        pb = policy_batches[pid]
        for col in (NODE_IDX, ADJ):
            if col not in pb:
                raise BatchError(f"batch of {pid!r} lacks column {col!r} (part of the Tuple observation)")
        if OBS not in pb:
            raise BatchError(f"batch of {pid!r} lacks column {OBS!r}")
        node, state, adj = check_graph_obs(pb[NODE_IDX], pb[OBS], pb[ADJ], pid)
        R = state.shape[0]
        cols = stack_policy_batches({pid: pb}, [pid], 0, self.A, TRAIN_COLUMNS[1:])
        if cols[ACTIONS].shape[1] != R:
            raise BatchError(f"{pid}: the train columns have {cols[ACTIONS].shape[1]} rows, the observation {R}")
        dev = lambda a: torch.from_numpy(a).to(self.device)
        d = {k: dev(v) for k, v in cols.items()}
        d.update({NODE_IDX: dev(node[None]), OBS: dev(state[None]), ADJ: dev(adj[None])})
        d, shuf, perms, used = self._prepare_batch(d, R, standardize)
        stats = self.learner.learn_on_batch(d[NODE_IDX][0], d[OBS][0], d[ADJ][0], d[ACTIONS][0], d[ACTION_DIST_INPUTS][0],
                                            d[ACTION_LOGP][0], d[VF_PREDS][0], d[ADVANTAGES][0], d[VALUE_TARGETS][0], perms[0],
                                            None if shuf is None else shuf[0], standardize=False)
        self.num_steps_trained += used
        return {pid: {"learner_stats": stats[0]}}

    # ---- weights ------------------------------------------------------------------------------------------------------
    def _weight_shapes(self):
        from .modelv2 import graphnet_shapes
        pid = self.policy_names[0]
        return [(f"{pid}/{name}", shp) for name, shp in graphnet_shapes(2 * self.A)]

    def get_weights(self) -> Dict[str, Dict[str, np.ndarray]]:
        """{pid: {"<pid>/actor/state_enc/kernel": ..., ..., "<pid>/critic/linear_out/bias": ...}}: the 12 variables of
        `modelv2.graphnet_shapes(2A)` in that order.  No reference checkpoint pins these names (no GraphNet checkpoint was
        published); they are the names the repository's ModelV2 class uses."""
        th = self.learner.theta.reshape(-1).cpu().numpy()
        out, o = {}, 0
        for name, shp in self._weight_shapes():
            n = int(np.prod(shp))
            out[name] = th[o:o + n].reshape(shp).copy()
            o += n
        return {self.policy_names[0]: out}

    def set_weights(self, weights: Mapping[str, Mapping[str, np.ndarray]]) -> None:
        """The inverse of `get_weights`: all 12 names with their exact shapes, nothing else (ValueError otherwise)."""
        import torch
        pid = self.policy_names[0]
        if pid not in weights:
            raise ValueError(f"set_weights: no weights for {pid!r}")
        w = weights[pid]
        want = self._weight_shapes()
        extra = sorted(set(w) - {name for name, _ in want})
        if extra:
            raise ValueError(f"set_weights: unknown variables {extra}")
        flat = []
        for name, shp in want:
            a = np.asarray(w[name], dtype=np.float32) if name in w else None
            if a is None or a.shape != tuple(shp):
                raise ValueError(f"set_weights: {name!r} of shape {tuple(shp)} is required, got "
                                 f"{None if a is None else a.shape}")
            flat.append(a.reshape(-1))
        self.learner.theta.copy_(torch.from_numpy(np.concatenate(flat)[None]).to(self.device))

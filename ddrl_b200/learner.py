"""Data-parallel PPO learner for the grouped per-leg controllers.

One learner iteration on a rollout ``[T, C]`` per policy (SURVEY.md §8-d):
  (i)   MeanStdFilter update + normalise, policy/value forward, DiagGaussian sample + logp   (K4, K1)
  (ii)  bootstrap value, GAE, advantage standardisation                                       (K1, K5)
  (iii) ``num_sgd_iter`` epochs of minibatch SGD.  Default (``mode="tc"``): ONE persistent tcgen05 launch per epoch
        that runs every optimizer step inside the kernel — forward + PPO loss + backward, fixed-order gradient
        reduction, in-kernel NVLink all-reduce over ranks, global-norm clip, TF1 Adam (csrc/tc2.cu, csrc/sgd_tail.cuh).
        ``mode="fp32"`` / ``fuse_tail=False`` keep the FP32-FMA kernel and the three-kernel step with an NCCL
        all-reduce between gradient reduce and Adam                                            (K2/K6, K7)
  (iv)  KL-coefficient update.
It replaces what RLlib 1.0.1 executes around the reference's models for ``tune.run("PPO", ...)``
(train_experiment_1_architecture_on_flat.py:201-211): sampler-side filter/forward, ``postprocess_ppo_gae``,
``StandardizeFields``, ``TrainTFMultiGPU`` and ``UpdateKL``.  All policies of an architecture are
processed by the same kernel launches ("grouped"); ranks shard the rollout by environment and exchange
only the flat gradient (every optimizer step), the filter partials, the advantage moments and the
learner-stat sums (once per iteration).

All arithmetic runs in libddrl_b200.so; torch provides memory, streams, CUDA graphs and the once-per-iteration NCCL
collectives (filter partials, advantage moments, stat sums)."""
from __future__ import annotations

import os
from typing import Dict, List, Optional

import numpy as np
import torch

from . import kernels as K
from ._lib import DDRLError, PPOHyper
from .config import PPOConfig
from .sharding import gather_stats_rank_order, local_minibatch

STAT_NAMES = ("total_loss", "policy_loss", "vf_loss", "kl", "entropy", "vf_explained_var")


def _dist_world():
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        return dist, dist.get_world_size(), dist.get_rank()
    return None, 1, 0


def finalize_stats(sums: np.ndarray, kl_coeff: np.ndarray, cfg: PPOConfig, rows: float) -> List[Dict[str, float]]:
    """sums [steps, P, 8] float64 (per-minibatch stat sums over ``rows`` global rows) -> per-policy learner
    stats averaged over the minibatches (float32 mean like RLlib's ``_averaged``)."""
    # All policies at once on [P, steps] arrays (the GPU idles while the host computes this between two iterations: 0.25 ms
    # per iteration when it was a per-policy loop of ~60 small numpy calls).  The float32 means run over the LAST, contiguous
    # axis, i.e. with the same pairwise summation as the 1-D means of the per-policy loop: identical bits.
    steps, P, _ = sums.shape
    n = float(rows)
    s = sums.transpose(1, 0, 2)                                      # [P, steps, 8] view
    pol, kl, vf, ent = s[..., 0] / n, s[..., 1] / n, s[..., 2] / n, s[..., 3] / n
    klc = np.asarray(kl_coeff, dtype=np.float64)[:P, None]
    total = pol + klc * kl + cfg.vf_loss_coeff * vf - cfg.entropy_coeff * ent
    yvar = s[..., 5] / n - (s[..., 4] / n) ** 2
    dvar = s[..., 7] / n - (s[..., 6] / n) ** 2
    with np.errstate(divide="ignore", invalid="ignore"):
        ev = np.maximum(-1.0, 1.0 - dvar / yvar)
    stacked = np.ascontiguousarray(np.stack([total, pol, vf, kl, ent, ev]).astype(np.float32))      # [6, P, steps]
    means = stacked.mean(axis=2).tolist()
    lr, ec = float(np.float32(cfg.lr)), float(cfg.entropy_coeff)
    return [{"total_loss": means[0][p], "policy_loss": means[1][p], "vf_loss": means[2][p], "kl": means[3][p],
             "entropy": means[4][p], "vf_explained_var": means[5][p], "cur_kl_coeff": float(np.float32(kl_coeff[p])),
             "cur_lr": lr, "entropy_coeff": ec} for p in range(P)]


_ENVELOPE = {"tc": "the tensor-core SGD step runs 1 <= D <= 63 and A in (1, 2, 4, 8)",
             "fp32": "the FP32 SGD step runs 1 <= D <= 64 and 1 <= A <= 8, with D <= 60 for A = 8 (shared memory)"}


def fcnet_mode_supports(D: int, A: int, mode: str) -> bool:
    """True if the SGD step of `mode` runs an FCNet of observation width D and action width A (ddrl_fcnet_train_supported)."""
    from . import _lib
    return bool(_lib.load().ddrl_fcnet_train_supported(int(D), int(A), int(mode == "tc")))


class _LearnerBase:
    def __init__(self, P: int, NP: int, cfg: PPOConfig, device, theta: Optional[torch.Tensor]):
        if not torch.cuda.is_available():
            raise DDRLError("ddrl_b200 learners need a CUDA device (sm_100a); there is no CPU fallback")
        self.P, self.NP, self.cfg = P, NP, cfg
        self.device = torch.device(device)
        f32 = torch.float32
        self.theta = (theta.to(self.device, f32).contiguous().clone() if theta is not None
                      else torch.zeros(P, NP, dtype=f32, device=self.device))
        if tuple(self.theta.shape) != (P, NP):
            raise DDRLError(f"theta shape {tuple(self.theta.shape)} != ({P}, {NP})")
        self.m = torch.zeros_like(self.theta)
        self.v = torch.zeros_like(self.theta)
        self.beta_pow = torch.tensor([[cfg.beta1, cfg.beta2]] * P, dtype=f32, device=self.device)
        self.kl_coeff_host = np.full(P, cfg.kl_coeff, dtype=np.float64)   # python-float state, like KLCoeffMixin.kl_coeff_val
        self.kl_coeff = torch.full((P,), cfg.kl_coeff, dtype=f32, device=self.device)
        self.grad = torch.zeros(P, NP, dtype=f32, device=self.device)
        self.gnorm = torch.zeros(P, dtype=f32, device=self.device)
        self.step_ctr = torch.zeros(1, dtype=torch.int32, device=self.device)
        self.sync_ws = torch.zeros(1, dtype=torch.int32, device=self.device)
        self.sync_token = torch.zeros(1, dtype=torch.float32, device=self.device)
        self.dist, self.world, self.rank = _dist_world()

    def _hyper(self, global_mb: int) -> PPOHyper:
        c = self.cfg
        return PPOHyper(c.clip_param, c.vf_clip_param, c.vf_loss_coeff, c.entropy_coeff, 1.0 / float(global_mb))

    def _adam(self):
        c = self.cfg
        img = getattr(self, "img", None)
        K.clip_adam(self.theta, self.m, self.v, self.beta_pow, self.grad, c.lr, c.beta1, c.beta2, c.adam_eps,
                    c.grad_clip, self.sync_ws, self.gnorm, self.step_ctr, img, getattr(self, "D", 0) if img is not None else 0,
                    self.A if img is not None else 0, tc_img=getattr(self, "tc_img", None))

    def standardize_advantages(self, adv: torch.Tensor) -> torch.Tensor:
        """StandardizeFields(["advantages"]) in place on adv [P,R] (float32, CUDA): per policy (adv - mean) / max(1e-4, std)
        over ALL rows of the train batch (all ranks' rows at world > 1).  The three moments are float64 torch reductions
        (plumbing); the rescale is `ddrl_adv_standardize`."""
        P = adv.shape[0]
        a64 = adv.reshape(P, -1).double()
        moments = torch.stack([torch.full((P,), float(a64.shape[1]), dtype=torch.float64, device=adv.device),
                               a64.sum(dim=1), (a64 * a64).sum(dim=1)], dim=1).contiguous()
        if self.world > 1:
            self.dist.all_reduce(moments)
        K.adv_standardize(adv, moments)
        return adv

    def _update_kl(self, stats: List[Dict[str, float]]):
        # KLCoeffMixin.update_kl (RLlib 1.0.1): x1.5 if kl > 2*target, x0.5 if kl < 0.5*target
        for p, s in enumerate(stats):
            if s["kl"] > 2.0 * self.cfg.kl_target:
                self.kl_coeff_host[p] *= 1.5
            elif s["kl"] < 0.5 * self.cfg.kl_target:
                self.kl_coeff_host[p] *= 0.5
        if getattr(self, "_kl_pinned", None) is None:
            try:
                self._kl_pinned = torch.empty(len(self.kl_coeff_host), dtype=torch.float32).pin_memory()
            except RuntimeError:      # no driver: host dry runs of the orchestration with mocked kernels (tests/test_host.py)
                self._kl_pinned = torch.empty(len(self.kl_coeff_host), dtype=torch.float32)
        # (pinned staging: the copy is queued without a host wait; the buffer is rewritten only after the next iteration's
        # stream synchronisation)
        self._kl_pinned.copy_(torch.from_numpy(self.kl_coeff_host.astype(np.float32)))
        self.kl_coeff.copy_(self._kl_pinned, non_blocking=True)


class FCNetLearner(_LearnerBase):
    """P grouped FCNet policies (obs dim D, action dim A, hiddens [64,64], tanh, separate value net)."""

    def __init__(self, P: int, D: int, A: int, cfg: PPOConfig, device="cuda", theta: Optional[torch.Tensor] = None,
                 use_graph: bool = True, ctas_per_policy: Optional[int] = None, mode: str = "tc", fuse_tail: bool = True,
                 persistent: bool = True, tc_forward: bool = True, ll_tail: bool = False, vf_share_layers: bool = False,
                 free_log_std: bool = False, atomic_reduce: bool = True, leg_coupling: bool = False):
        """mode: "tc"   = tensor-core (tcgen05) SGD step, fp16 hi/lo operand split (gradients within 5e-5 of scale);
                 "fp32" = FP32-FMA SGD step (1e-5 parity).  Inference / GAE / Adam are FP32 in both modes.
        vf_share_layers / free_log_std: the reference model's optional layouts (models/fcnet_glorot_uniform_init.py:30-36,
        85-113).  `theta` is then [P, NPm] in the MODEL's variable order (`modelv2.fcnet_variant_shapes`); the kernels run on
        its index-select (`self.theta`, tied value branch / constant zero columns), the gradients of tied copies are added
        (`ddrl_grad_tie`) and clip + Adam act on the model variables (`self.theta_model`) — the kernel-per-stage step, since
        the fused tail owns kernel-layout slices.
        leg_coupling: the policy of QuantrupedMultiEnv_SharedDecentralLegID (model "cup" = FCNet + LegCoupling,
        models/coupling_net_glorot_uniform_init.py:11-30,135): ONE shared policy (P = 1), A = 2.  `theta` is then
        [1, NP + 8] — the 12 FCNet variables in checkpoint order, then leg_coupling [4, 2] row-major (the registration order
        of the ModelV2 class); m / v alike; default table LegCoupling.INIT.  The mean logits of a row are scaled by
        c[node id], node id = the agent's position in agent_names (FL, HL, HR, FR); the SGD steps are
        ddrl_ppo_train_step_tc_coupled / ddrl_ppo_train_step_coupled (fused tail required: the table is clipped and stepped
        with the MLP weights)."""
        if mode not in ("tc", "fp32"):
            raise DDRLError(f"mode must be 'tc' or 'fp32', got {mode!r}")
        if not fcnet_mode_supports(D, A, mode):
            raise DDRLError(f"mode={mode!r} cannot train an FCNet with D={D}, A={A}: " + _ENVELOPE[mode])
        self.coupled = bool(leg_coupling)
        if self.coupled:
            if P != 1 or A != 2:
                raise DDRLError(f"leg_coupling: the coupled model is one shared policy with A = 2 (got P={P}, A={A})")
            if not fuse_tail or ll_tail or vf_share_layers or free_log_std:
                raise DDRLError("leg_coupling: fuse_tail=False, ll_tail and the optional FCNet layouts are not supported")
            if mode == "tc" and D not in (19, 20):
                raise DDRLError(f"leg_coupling: the tensor-core step is instantiated for D in (19, 20), got D={D}")
            if _dist_world()[1] > 1:
                raise DDRLError("leg_coupling: data-parallel training (world > 1) is not supported")
            if theta is None:
                theta = torch.zeros(1, K.fcnet_num_params(D, A) + 8, dtype=torch.float32)
                from .modelv2 import LegCoupling
                theta[0, -8:] = torch.tensor(LegCoupling.INIT, dtype=torch.float32).reshape(-1)
        self.variant = bool(vf_share_layers or free_log_std)
        theta_model = None
        if self.variant:
            from .modelv2 import fcnet_layout_map, fcnet_variant_shapes
            lmap = fcnet_layout_map(D, 2 * A, vf_share_layers, free_log_std)
            NPm = int(sum(int(np.prod(shp)) for _, shp in fcnet_variant_shapes(D, 2 * A, vf_share_layers, free_log_std)))
            if theta is None or tuple(theta.shape) != (P, NPm):
                raise DDRLError(f"optional FCNet layout: theta must be [P={P}, {NPm}] in the model's variable order")
            theta_model, theta = theta, None
            fuse_tail, persistent = False, False
        self.NPf = K.fcnet_num_params(D, A)      # FCNet variables (the coupled model adds its table behind them)
        super().__init__(P, self.NPf + (8 if self.coupled else 0), cfg, device, theta)
        self.theta_fc = self.theta[:, :self.NPf]      # (view: the FCNet part, what the weight images are packed from)
        if self.variant:
            dev_ = self.device
            self.NPm = NPm
            self.theta_model = theta_model.to(dev_, torch.float32).contiguous().clone()
            self.m = torch.zeros_like(self.theta_model)
            self.v = torch.zeros_like(self.theta_model)
            self.grad_model = torch.zeros_like(self.theta_model)
            self.layout_map = lmap.to(torch.int32).to(dev_)
            inv = torch.full((NPm, 2), -1, dtype=torch.int32)
            for i, j in enumerate(lmap.tolist()):
                if j < NPm:
                    inv[j, 0 if inv[j, 0] < 0 else 1] = i
            self.inverse_map = inv.to(dev_)
            K.param_expand(self.theta_model, self.layout_map, self.theta)
        self.mode = mode
        self.fuse_tail = fuse_tail
        self.persistent = persistent      # one persistent launch per epoch where the kernel supports it
        self.tc_forward = tc_forward and mode == "tc"   # inference forward on the tensor cores as well
        # opt-in: the CTAs hand their partial gradients to the slice owners as self-validating {payload, tag} words pulled
        # with TMA bulk copies instead of plain arrays behind barrier A (csrc/sgd_tail.cuh).  Measured on the bench workload:
        # 30.3 us per step against 29.4 us for the three-barrier tail (the 8-byte words double the early write-out), so
        # it is OFF by default; DDRL_LL_TAIL=1 switches it on for A/B timing
        self.ll_tail = (ll_tail or os.environ.get("DDRL_LL_TAIL", "0") == "1") and mode == "tc"
        # the CTAs of a policy ADD their partial gradients into one vector at L2 (red.global.add.v4.f32) instead of writing G
        # partials that every slice owner reads back: 1.4 us per step faster on the bench workload, but the order of the float
        # additions is no longer fixed (last-bit differences from run to run; the ranks of one run still end bit-identical).
        # atomic_reduce=False / DDRL_FIXED_ORDER=1 keeps the fixed-order, bit-reproducible reduction
        self.atomic_reduce = (atomic_reduce and os.environ.get("DDRL_FIXED_ORDER", "0") != "1" and mode == "tc"
                              and not self.ll_tail)
        self.D, self.A = D, A
        dev = self.device
        self.filt_n = torch.zeros(P, dtype=torch.int64, device=dev)
        self.filt_M = torch.zeros(P, D, dtype=torch.float64, device=dev)
        self.filt_S = torch.zeros(P, D, dtype=torch.float64, device=dev)
        self.norm = torch.zeros(P, 2, D, dtype=torch.float64, device=dev)
        self._filt_tmp = {"n": torch.zeros(P, dtype=torch.int64, device=dev), "M": torch.zeros(P, D, dtype=torch.float64, device=dev),
                          "S": torch.zeros(P, D, dtype=torch.float64, device=dev),
                          "norm": torch.zeros(P, 2, D, dtype=torch.float64, device=dev)}      # per-rank merge at world > 1
        self.use_graph = use_graph
        self.ctas_per_policy = ctas_per_policy
        # packed shared-memory image of the weights (kept in step by clip_adam); rebuilt at every iteration start so
        # external writes to self.theta (checkpoint import) are picked up
        self.img = torch.zeros(P, K.fcnet_image_floats(D, A), dtype=torch.float32, device=dev)
        self.tc_img = None
        self.tc_status = torch.zeros(1, dtype=torch.int32, device=dev)
        if mode == "tc":
            self.tc_img = K.fcnet_tc_pack(self.theta_fc, D, A)
        self._bufs = None
        self._graph = None
        self._graph_key = None
        self.sms = torch.cuda.get_device_properties(dev).multi_processor_count
        self._peers = None
        self._prep_graphs = {}
        self._prep_warm = False

    # ---- buffers ------------------------------------------------------------------------------------
    def _alloc(self, T: int, Cc: int):
        key = (T, Cc)
        if self._bufs is not None and self._bufs["key"] == key:
            return self._bufs
        P, D, A, dev, f32 = self.P, self.D, self.A, self.device, torch.float32
        R = T * Cc
        b = {"key": key}
        for name, w in (("obs", D), ("act", A), ("logits", 2 * A)):
            b[name] = torch.empty(P, R, w, dtype=f32, device=dev)
            b[name + "_s"] = torch.empty(P, R, w, dtype=f32, device=dev)
        for name in ("logp", "value", "adv", "vtarg"):
            b[name] = torch.empty(P, R, dtype=f32, device=dev)
            b[name + "_s"] = torch.empty(P, R, dtype=f32, device=dev)
        b["vboot"] = torch.empty(P, Cc, dtype=f32, device=dev)
        if self.coupled:      # node id of every row (learn_on_rollout: column c of an env-major [T, C] rollout is leg c % 4)
            b["node"] = (torch.arange(R, dtype=torch.int32, device=dev) % 4).reshape(1, R).contiguous()
            b["node_s"] = torch.empty_like(b["node"])
        b["moments"] = torch.empty(P, 3, dtype=torch.float64, device=dev)
        b["gae_ws"] = torch.empty(max(8, P * ((Cc + 255) // 256) * 16), dtype=torch.uint8, device=dev)
        b["filt_ws"] = None
        self._bufs = b
        self._graph = None
        return b

    def _sgd_setup(self, R: int):
        cfg, P = self.cfg, self.P
        MB = min(local_minibatch(cfg.sgd_minibatch_size, self.world), R)
        if MB < 1:
            raise DDRLError("sgd_minibatch_size smaller than the number of ranks")
        nb = max(1, R // MB)
        G = self.ctas_per_policy or max(1, min((MB + 15) // 16, self.sms // P))
        if not self.ctas_per_policy and self.mode == "tc" and self.fuse_tail and self.sms // P >= 32:
            # measured (profiles/README.md, CTA sweep): the fused tail (three barriers among the G CTAs of a policy, one
            # parameter slice per CTA) is fastest around G = 32 whatever the minibatch size, as long as no CTA needs an
            # extra 128-row tile for it; CTAs without rows still own a slice
            tiles = lambda g: -(-((-(-MB // g) + 7) // 8 * 8) // 128)
            if tiles(32) <= tiles(self.sms // P):
                G = 32
        return MB, nb, G

    # ---- one optimizer step (3 kernels [+ NCCL]) -----------------------------------------------------------
    def _peer_exchange(self, G: int):
        """Peer-mapped exchange buffers of the in-kernel gradient all-reduce (world > 1), created once per shape."""
        key = (self.P, self.NP, G)
        if self._peers is None or self._peers.key != key:
            from .peer import PeerExchange
            if self._peers is not None:
                self._peers.close()
            self._peers = PeerExchange(self.dist, self.world, self.rank, self.P, self.NP, G, self.device)
        return self._peers

    def _sgd_step(self, b, MB, G, hyper, src, nsteps: int = 1):
        # ONE launch per optimizer step: the train kernel also reduces the partials, all-reduces the gradient slices
        # over NVLink peer memory (world > 1), clips and applies Adam (csrc/sgd_tail.cuh).  With nsteps > 1 (ping-pong
        # tcgen05 kernel) ONE persistent launch runs that many consecutive steps.  fuse_tail=False keeps the 3-kernel
        # path (train, grad_reduce, [NCCL all-reduce], clip_adam) for A/B tests.
        tail = None
        if self.fuse_tail and G * self.P <= self.sms:
            c = self.cfg
            # the descriptor only holds pointers and hyper-parameters: built once per buffer set (the host work between two
            # iterations is exposed GPU idle time: tests/iter_breakdown.py)
            key = (b["tail_bar"].data_ptr(), b["step_stats"].data_ptr(), G, self.mode, c.lr, c.grad_clip)
            cached = b.get("tail_desc")
            if cached is None or cached[0] != key:
                tail = K.make_sgd_tail(self.theta, self.m, self.v, self.beta_pow, self.grad, b["tail_bar"], b["tail_sq"], c.lr,
                                       c.beta1, c.beta2, c.adam_eps, c.grad_clip, self.gnorm,
                                       img=self.img if self.mode == "fp32" else None, tc_img=self.tc_img,
                                       step_stats=b["step_stats"], step_ctr=self.step_ctr, status=self.tc_status,
                                       ll_ws=b.get("tail_ll"), grad_acc=b.get("tail_acc"))
                b["tail_desc"] = (key, tail)
            else:
                tail = cached[1]
            tail.nsteps = nsteps
            if self.world > 1:
                self._peer_exchange(G).fill(tail)
        elif nsteps != 1:
            raise DDRLError("multi-step launches need the fused tail")
        if self.coupled and tail is None:
            raise DDRLError("leg_coupling: the coupled SGD step needs the fused tail")
        batch = (src["obs"], src["act"], src["logits"], src["logp"], src["value"], src["adv"], src["vtarg"], self.A, MB,
                 b["mb_perm"], self.step_ctr, self.kl_coeff, hyper, G, b["grad_part"], b["stat_part"])
        if self.mode == "tc" and self.coupled:
            K.ppo_train_step_tc_coupled(self.tc_img, self.theta, src["node"], *batch, self.tc_status, tail)
        elif self.mode == "tc":
            K.ppo_train_step_tc(self.tc_img, *batch, self.tc_status, tail=tail)
        elif self.coupled:
            K.ppo_train_step_coupled(self.theta, self.img, src["node"], *batch, tail)
        else:
            K.ppo_train_step(self.theta, *batch, img=self.img, tail=tail)
        if tail is not None:
            return
        K.grad_reduce(b["grad_part"], b["stat_part"], self.P, G, self.NP, self.grad, b["step_stats"], self.step_ctr)
        if self.variant:
            # optional layouts: tie the gradients of the copies, clip + Adam on the MODEL's variables, re-expand, re-pack
            c = self.cfg
            K.grad_tie(self.grad, self.inverse_map, self.grad_model)
            if self.world > 1:
                self.dist.all_reduce(self.grad_model)
            K.clip_adam(self.theta_model, self.m, self.v, self.beta_pow, self.grad_model, c.lr, c.beta1, c.beta2, c.adam_eps,
                        c.grad_clip, self.sync_ws, self.gnorm, self.step_ctr, None, 0, 0)
            K.param_expand(self.theta_model, self.layout_map, self.theta)
            K.fcnet_pack(self.theta, self.D, self.A, self.img)
            if self.tc_img is not None:
                K.fcnet_tc_pack(self.theta, self.D, self.A, self.tc_img)
            return
        if self.world > 1:
            self.dist.all_reduce(self.grad)
        self._adam()

    def _persistent_steps(self, G: int) -> bool:
        """True if one launch can run a whole epoch of SGD steps (ping-pong tcgen05 kernel + fused tail)."""
        return (self.persistent and self.mode == "tc" and self.fuse_tail and G * self.P <= self.sms
                and K.tc_pingpong_eligible(self.D, self.A))

    # ---- everything before the SGD epochs: filter, inference forward, bootstrap, GAE, standardise, shuffle ----------------
    def _prepare(self, b, obs_flat, boot_obs, rewards, dones, eps_flat, shuffle, cols_per_env, update_filter, T, Cc):
        P, R, D = obs_flat.shape
        cfg = self.cfg
        self.tc_status.zero_()
        self._pack_images()
        # (i) filter + forward + sample ------------------------------------------------------------------
        if update_filter:
            if self.world > 1:
                # this rank's partials -> ONE {count, mean, M2} per (policy, feature) (Chan merge into a zero state), the
                # ranks' triples gathered in rank order, then folded into the running state: identical bits on every rank
                t = self._filt_tmp
                for k in ("n", "M", "S"):
                    t[k].zero_()
                K.filter_merge(K.filter_partial(obs_flat), R, t["n"], t["M"], t["S"], t["norm"])
                one = torch.stack([t["n"].double().unsqueeze(1).expand(P, D), t["M"], t["S"]], dim=-1).reshape(P, 1, D, 3)
                allp = gather_stats_rank_order(one, self.dist, self.world)
                K.filter_merge(allp, R * self.world, self.filt_n, self.filt_M, self.filt_S, self.norm)
            else:
                K.filter_update(obs_flat, self.filt_n, self.filt_M, self.filt_S, self.norm, b["filt_ws"])
        # the rollout rows (coupled: the stored old logits are the COUPLED ones), then the bootstrap values
        self._forward(obs_flat, {"logits": b["logits"], "value": b["value"], "obs_out": b["obs"], "action": b["act"],
                                 "logp": b["logp"]}, eps=eps_flat, node=b["node"] if self.coupled else None)
        self._forward(boot_obs, {"logits": None, "value": b["vboot"], "obs_out": None})
        # (ii) bootstrap + GAE + standardise -----------------------------------------------------------
        K.gae(rewards, b["value"].view(P, T, Cc), dones, b["vboot"], cols_per_env, cfg.gamma, cfg.lambda_,
              b["adv"].view(P, T, Cc), b["vtarg"].view(P, T, Cc), b["moments"], b["gae_ws"])
        if self.world > 1:
            self.dist.all_reduce(b["moments"])
        K.adv_standardize(b["adv"], b["moments"])
        if shuffle is not None:
            self._shuffle(b, shuffle)

    _COLUMNS = ("obs", "act", "logits", "logp", "value", "adv", "vtarg")

    def _pack_images(self):
        """The FP32 and tensor-core weight images, from the FCNet part of theta."""
        K.fcnet_pack(self.theta_fc, self.D, self.A, self.img)
        if self.tc_img is not None:
            K.fcnet_tc_pack(self.theta_fc, self.D, self.A, self.tc_img)

    def _shuffle(self, b, shuffle):
        """SampleBatch.shuffle: the columns, row-permuted into their *_s buffers."""
        for nme in self._COLUMNS:
            K.gather_rows(b[nme], shuffle, b[nme + "_s"])
        if self.coupled:      # the node ids travel with their rows (a 4-byte row copy: the int32 bits move unchanged)
            K.gather_rows(b["node"].view(torch.float32), shuffle, b["node_s"].view(torch.float32))

    def _src(self, b, shuffled: bool) -> dict:
        """The columns the SGD phase reads: the shuffled *_s buffers or the prepared ones."""
        names = self._COLUMNS + (("node",) if self.coupled else ())
        return {n_: b[n_ + ("_s" if shuffled else "")] for n_ in names}

    def _forward(self, obs, out: dict, eps=None, node=None):
        """Inference forward of rows `obs` into `out` (filter normalisation with self.norm; with eps the DiagGaussian sample).
        With `node` the leg-coupled model in ONE launch: forward, LegCoupling on the mean logits, sample + logp of the
        coupled distribution.  On the tensor cores if tc_forward (same pipeline as the training forward, ~3e-6 relative) —
        the uncoupled model only where the ping-pong kernel runs its shape — else on the FP32 kernel."""
        kw = dict(norm=self.norm, clip=self.cfg.filter_clip, eps=eps, out=out)
        tc = self.tc_forward and (self.coupled or K.tc_pingpong_eligible(self.D, self.A))
        if node is not None:
            coupling = self.theta[0, self.NPf:]
            if tc:
                K.fcnet_forward_tc_coupled(self.tc_img, obs, node, coupling, self.A, status=self.tc_status, **kw)
            else:
                K.fcnet_forward_coupled(self.theta_fc, obs, node, coupling, self.A, status=self.tc_status, img=self.img, **kw)
        elif tc:
            K.fcnet_forward_tc(self.tc_img, obs, self.A, status=self.tc_status, **kw)
        else:
            K.fcnet_forward(self.theta_fc, obs, self.A, img=self.img, **kw)

    def _prepare_cached(self, b, obs_flat, boot_obs, rewards, dones, eps_flat, shuffle, cols_per_env, update_filter, T, Cc):
        """The ~20 short launches of the preparation phase are captured once per set of input buffers and replayed (the
        kernels only see pointers; graphs are keyed by the input addresses, at most 8 are kept).  At world > 1 the capture
        includes the three NCCL collectives of the phase (filter partials, advantage moments); every rank captures and
        replays in the same iteration, so the collectives stay matched."""
        args = (b, obs_flat, boot_obs, rewards, dones, eps_flat, shuffle, cols_per_env, update_filter, T, Cc)
        if not self.use_graph or self._prep_graphs is None or not self._prep_warm:
            self._prep_warm = True           # first call runs eagerly (one-time function attributes, lazy allocations)
            return self._prepare(*args)
        if b.get("filt_ws") is None:
            from . import _lib
            nbytes = int(_lib.load().ddrl_filter_ws_bytes(obs_flat.shape[0], obs_flat.shape[1], obs_flat.shape[2]))
            b["filt_ws"] = torch.empty(max(nbytes, 8), dtype=torch.uint8, device=self.device)
        key = (obs_flat.data_ptr(), boot_obs.data_ptr(), rewards.data_ptr(), dones.data_ptr(), eps_flat.data_ptr(),
               shuffle.data_ptr() if shuffle is not None else 0, tuple(obs_flat.shape), cols_per_env, bool(update_filter), id(b))
        g = self._prep_graphs.get(key)
        if g is None:
            if len(self._prep_graphs) >= 8:      # inputs keep moving (fresh tensors every call): stop capturing
                self._prep_graphs = None
                return self._prepare(*args)
            try:
                torch.cuda.synchronize()
                if self.world > 1:
                    self.dist.barrier()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    self._prepare(*args)
                self._prep_graphs[key] = g
            except Exception as exc:
                self._prep_graphs = None
                self.graph_error = repr(exc)
                torch.cuda.synchronize()
                return self._prepare(*args)
        g.replay()

    # ---- the iteration --------------------------------------------------------------------------------------
    def learn_on_rollout(self, raw_obs: torch.Tensor, boot_obs: torch.Tensor, rewards: torch.Tensor,
                         dones: torch.Tensor, eps: torch.Tensor, perms: torch.Tensor,
                         shuffle: Optional[torch.Tensor] = None, cols_per_env: int = 1,
                         update_filter: bool = True) -> List[Dict[str, float]]:
        """raw_obs [P,T,C,D] f32 (index-gathered per policy), boot_obs [P,C,D], rewards [P,T,C], dones [T,C/cpe] u8,
        eps [P,T,C,A] (N(0,1) noise for action sampling), perms [P,E,nb] int32 (minibatch visiting order per epoch,
        np.random.permutation(nb) in RLlib), shuffle [P,T*C] int32 row permutation or None.  All CUDA tensors.
        Returns the per-policy learner stats of the LAST epoch and updates weights / Adam / filter / kl_coeff."""
        P, T, Cc, D = raw_obs.shape
        cfg, A = self.cfg, self.A
        if D != self.D or P != self.P:
            raise DDRLError(f"raw_obs shape {tuple(raw_obs.shape)} does not match learner (P={self.P}, D={self.D})")
        R = T * Cc
        if self.coupled and (cols_per_env != 4 or Cc % 4):
            raise DDRLError(f"leg_coupling: the rollout's columns must be env-major legs (cols_per_env=4, C % 4 == 0), got "
                            f"cols_per_env={cols_per_env}, C={Cc}")
        b = self._alloc(T, Cc)
        obs_flat = raw_obs.reshape(P, R, D)
        eps_flat = eps.reshape(P, R, A)
        self._prepare_cached(b, obs_flat, boot_obs, rewards, dones, eps_flat, shuffle, cols_per_env, update_filter, T, Cc)
        return self._sgd_phase(b, self._src(b, shuffle is not None), "s" if shuffle is not None else "u", perms, R, T, Cc)

    def _sgd_phase(self, b, src, src_key, perms, R: int, T: int, Cc: int) -> List[Dict[str, float]]:
        """(iii) minibatch SGD over the prepared columns `src` + (iv) stats and KL-coefficient update."""
        P, cfg = self.P, self.cfg
        E = perms.shape[1]
        MB, nb, G = self._sgd_setup(R)
        if perms.shape[2] != nb:
            raise DDRLError(f"perms has {perms.shape[2]} minibatches per epoch, expected {nb} (R={R}, MB={MB})")
        steps = E * nb
        if b.get("sgd_key") != (steps, G):
            b["sgd_key"] = (steps, G)
            b["mb_perm"] = torch.empty(P, steps, dtype=torch.int32, device=self.device)
            b["grad_part"] = torch.empty(P, G, K.part_stride(self.NP), dtype=torch.float32, device=self.device)
            b["stat_part"] = torch.empty(P, G, K.NSTAT, dtype=torch.float64, device=self.device)
            b["step_stats"] = torch.zeros(steps, P, K.NSTAT, dtype=torch.float64, device=self.device)
            b["tail_bar"] = torch.zeros(4 * P + 4, dtype=torch.int32, device=self.device)
            b["tail_sq"] = torch.zeros(P, G, 32, dtype=torch.float32, device=self.device)   # one 128-byte line per {sum, tag} word
            # LL workspace: same lifetime as tail_bar (its tags are the step count kept there)
            b["tail_ll"] = (torch.zeros(K.sgd_ll_words(P, G, self.D, self.A), dtype=torch.int64, device=self.device)
                            if self.ll_tail and K.tc_pingpong_eligible(self.D, self.A) else None)
            b["tail_acc"] = (torch.zeros(P, K.part_stride(self.NP), dtype=torch.float32, device=self.device)
                             if self.atomic_reduce and K.tc_pingpong_eligible(self.D, self.A) else None)
            self._graph = None
        b["mb_perm"].copy_(perms.reshape(P, steps))
        self.step_ctr.zero_()
        hyper = self._hyper(MB * self.world)
        if self.world > 1:
            # the persistent kernels exchange gradients over peer memory with BOUNDED spins: line the ranks' streams up first
            # (one tiny collective; learn_on_batch(standardize=False) has no other collective ahead of the launch)
            self.dist.all_reduce(self.sync_token)
        if self.world > 1 and self.fuse_tail and G * P <= self.sms:
            self._peer_exchange(G)      # allocate / map the peer buffers outside any graph capture
        ran = False
        if self._persistent_steps(G):
            # ONE persistent launch for the whole SGD phase: all E * nb optimizer steps run inside the kernel (the minibatch
            # order of every epoch is in mb_perm; no graph needed)
            self._sgd_step(b, MB, G, hyper, src, nsteps=steps)
            ran = True
        elif self.use_graph:
            key = (T, Cc, steps, G, MB, src_key)
            if self._graph is None or self._graph_key != key:
                torch.cuda.synchronize()
                if self.world > 1:
                    self.dist.barrier()
                try:
                    g = torch.cuda.CUDAGraph()
                    # the capture executes nothing; kernels read step_ctr / mb_perm / kl_coeff from device memory, so
                    # one captured epoch (nb steps incl. the NCCL all-reduce at N>1) serves every epoch and iteration
                    with torch.cuda.graph(g):
                        for _ in range(nb):
                            self._sgd_step(b, MB, G, hyper, src)
                    self._graph, self._graph_key = g, key
                    if self.world > 1:
                        self.dist.barrier()     # replays spin on peer flags: start them together
                except Exception as exc:  # capture not possible (e.g. NCCL build without graph support): run eagerly
                    self._graph, self.use_graph = None, False
                    self.graph_error = repr(exc)
                    torch.cuda.synchronize()
                    self.step_ctr.zero_()
            if self._graph is not None:
                for _ in range(E):
                    self._graph.replay()
                ran = True
        if not ran:
            for _ in range(steps):
                self._sgd_step(b, MB, G, hyper, src)
        # (iv) stats + KL update ----------------------------------------------------------------------------
        if self.world > 1:
            last = b["step_stats"][steps - nb:].clone()
            self.dist.all_reduce(last)
            sums = last.cpu().numpy()
            code = int(self.tc_status.item())
        else:
            # ONE host round trip: both reads go to pinned memory behind the SGD phase, one stream synchronisation
            hb = b.get("host_stats")
            if hb is None or tuple(hb.shape) != (nb, P, K.NSTAT):
                hb = b["host_stats"] = torch.empty(nb, P, K.NSTAT, dtype=torch.float64).pin_memory()
                b["host_status"] = torch.zeros(1, dtype=torch.int32).pin_memory()
            hb.copy_(b["step_stats"][steps - nb:], non_blocking=True)
            b["host_status"].copy_(self.tc_status, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            sums = hb.numpy()
            code = int(b["host_status"][0])
        stats = finalize_stats(sums, self.kl_coeff_host, cfg, MB * self.world)
        if code:
            what = [n for bit, n in ((1, "MMA completion timed out"), (2, "x overflow"), (4, "activation overflow"),
                                     (8, "dl overflow"), (16, "dz2 overflow"), (32, "dz1 overflow"),
                                     (64, "fused-tail barrier / peer wait timed out"),
                                     (K.STATUS_BAD_NODE, "leg-coupling node id outside 0..3")) if code & bit]
            fp32 = ("use mode='fp32' for this workload" if fcnet_mode_supports(self.D, self.A, "fp32") else
                    f"mode='fp32' cannot train this shape either ({_ENVELOPE['fp32']})")
            hint = (" — fp16 split range exceeded: " + fp32 if code & 62 else
                    " — node ids must be 0..3 (FL, HL, HR, FR)" if code & K.STATUS_BAD_NODE else
                    " — a CTA barrier or a peer rank did not arrive in time")
            raise DDRLError("SGD step failed (" + ", ".join(what) + ")" + hint)
        self._update_kl(stats)
        return stats

    def learn_on_batch(self, obs: torch.Tensor, actions: torch.Tensor, action_dist_inputs: torch.Tensor,
                       action_logp: torch.Tensor, vf_preds: torch.Tensor, advantages: torch.Tensor,
                       value_targets: torch.Tensor, perms: torch.Tensor, shuffle: Optional[torch.Tensor] = None,
                       standardize: bool = True, node_idx: Optional[torch.Tensor] = None) -> List[Dict[str, float]]:
        """The learner half only, on POSTPROCESSED sample-batch columns as RLlib's `Policy.learn_on_batch` receives them
        (rollout workers have already filtered the observations, sampled the actions and run `postprocess_ppo_gae`):
        obs [P,R,D] (filtered), actions [P,R,A], action_dist_inputs [P,R,2A], action_logp / vf_preds / advantages /
        value_targets [P,R] — float32 CUDA tensors, one row block per policy.  `standardize` applies
        StandardizeFields(["advantages"]) per policy; `shuffle` [P,R] int32 and `perms` [P,E,nb] as in learn_on_rollout.
        Runs StandardizeFields -> shuffle -> E x nb minibatch steps -> KL update and returns the learner stats.
        leg_coupling: node_idx [1,R] int32 CUDA (0..3: FL, HL, HR, FR) is required; action_dist_inputs are coupled logits."""
        P, R, D = obs.shape
        A = self.A
        if D != self.D or P != self.P:
            raise DDRLError(f"obs shape {tuple(obs.shape)} does not match learner (P={self.P}, D={self.D})")
        if self.coupled != (node_idx is not None):
            raise DDRLError("learn_on_batch: node_idx [1, R] int32 is required with leg_coupling and only then")
        if node_idx is not None and (tuple(node_idx.shape) != (P, R) or node_idx.dtype != torch.int32 or not node_idx.is_cuda):
            raise DDRLError(f"learn_on_batch: node_idx must be an int32 CUDA tensor of shape {(P, R)}, got {node_idx.dtype} "
                            f"{tuple(node_idx.shape)} on {node_idx.device}")
        cols = {"obs": (obs, (P, R, D)), "act": (actions, (P, R, A)), "logits": (action_dist_inputs, (P, R, 2 * A)),
                "logp": (action_logp, (P, R)), "value": (vf_preds, (P, R)), "adv": (advantages, (P, R)),
                "vtarg": (value_targets, (P, R))}
        for name, (t, shape) in cols.items():
            if tuple(t.shape) != shape or t.dtype != torch.float32 or not t.is_cuda:
                raise DDRLError(f"learn_on_batch: column {name!r} must be a float32 CUDA tensor of shape {shape}, "
                                f"got {t.dtype} {tuple(t.shape)} on {t.device}")
        b = self._alloc(R, 1)
        self.tc_status.zero_()
        self._pack_images()
        for name, (t, _) in cols.items():
            b[name].copy_(t)
        if self.coupled:
            b["node"].copy_(node_idx)
        if standardize:
            self.standardize_advantages(b["adv"])
        if shuffle is not None:
            self._shuffle(b, shuffle)
        return self._sgd_phase(b, self._src(b, shuffle is not None), "s" if shuffle is not None else "u", perms, R, R, 1)

    def refresh_filter_norm(self):
        """Recompute the normalisation table (mean, 1/(std+1e-8)) from filt_n / filt_M / filt_S — after the state was
        written from outside (checkpoint import)."""
        zero = torch.zeros(self.P, 1, self.D, 3, dtype=torch.float64, device=self.device)
        K.filter_merge(zero, 0, self.filt_n, self.filt_M, self.filt_S, self.norm)

    # ---- plain inference (sampler side) ---------------------------------------------------------------------
    def compute_actions(self, raw_obs: torch.Tensor, eps: Optional[torch.Tensor] = None, update_filter: bool = False,
                        node_idx: Optional[torch.Tensor] = None):
        """raw_obs [P,B,D] -> dict(logits, value[, action, logp]); optionally pushes the rows into the filter first
        (RLlib sampler behaviour).  leg_coupling: node_idx [1,B] int32 (required); logits / action / logp are those of the
        coupled distribution."""
        if self.coupled != (node_idx is not None):
            raise DDRLError("compute_actions: node_idx [1, B] int32 is required with leg_coupling and only then")
        if update_filter:
            K.filter_update(raw_obs, self.filt_n, self.filt_M, self.filt_S, self.norm)
        use_norm = self.norm if int(self.filt_n.max().item()) > 0 else None
        if not self.coupled:
            return K.fcnet_forward(self.theta, raw_obs, self.A, norm=use_norm, clip=self.cfg.filter_clip, eps=eps)
        P, B, _ = raw_obs.shape
        if tuple(node_idx.shape) != (P, B) or node_idx.dtype != torch.int32 or not node_idx.is_cuda:
            raise DDRLError(f"compute_actions: node_idx must be an int32 CUDA tensor of shape {(P, B)}")
        res = K.fcnet_forward_coupled(self.theta_fc, raw_obs, node_idx.contiguous(), self.theta[0, self.NPf:], self.A,
                                      norm=use_norm, clip=self.cfg.filter_clip, eps=eps)
        if int(res.pop("status").item()) & K.STATUS_BAD_NODE:
            raise DDRLError("compute_actions: node ids must be 0..3 (FL, HL, HR, FR)")
        res.pop("obs_out")
        return res


class GraphNetLearner(_LearnerBase):
    """One shared GraphNet policy (actor GraphNet(2A) + critic GraphNet(1)) over the 4-leg graph
    (models/shared_graphnet_glorot_uniform_init.py:21-58; env QuantrupedMultiEnv_DecentralShared_Graph).
    The observations reach the model already normalised (the env-side filter runs before the tuple is built,
    quantruped_GraphDecentralizedController_environments.py:219-233), so there is no filter stage here."""

    def __init__(self, A: int, cfg: PPOConfig, device="cuda", theta: Optional[torch.Tensor] = None,
                 ctas: Optional[int] = None, two_launch_step: bool = False, step: Optional[str] = None):
        """step: "tc" (default) = ONE persistent launch per epoch, `ddrl_graphnet_train_step_tc`: FMA/MUFU hyper-encoder,
        tcgen05 MPNN / head / weight-gradient GEMMs, fused gradient reduce + in-kernel NVLink all-reduce + clip + Adam;
        "three-kernel" = forward + ppo_loss_grad + row-per-CTA backward + reduce + Adam (FP32, 1e-5 path, A/B reference);
        "two-launch" (or two_launch_step=True) = `ddrl_graphnet_train_step` (measured slower than three-kernel)."""
        super().__init__(1, K.graphnet_num_params(2 * A), cfg, device, theta)
        self.A = A
        self.step_kind = step or ("two-launch" if two_launch_step else os.environ.get("DDRL_GN_STEP", "tc"))
        if self.step_kind not in ("tc", "three-kernel", "two-launch"):
            raise DDRLError(f"GraphNetLearner: unknown step kind {self.step_kind!r}")
        self.two_launch_step = self.step_kind == "two-launch"
        self.sms = torch.cuda.get_device_properties(self.device).multi_processor_count
        self.ctas = ctas or max(1, self.sms // 2)
        self.status = torch.zeros(1, dtype=torch.int32, device=self.device)
        self._tc = None
        self._peers = None

    def forward(self, node_idx, state, adj):
        return K.graphnet_forward(self.theta.reshape(-1), node_idx, state, adj, self.A)

    # ---- plain inference (sampler side) ---------------------------------------------------------------------
    def compute_actions(self, node_idx: torch.Tensor, state: torch.Tensor, adj: torch.Tensor,
                        eps: Optional[torch.Tensor] = None):
        """node_idx [B] int32 (0..3: FL, HL, HR, FR), state [B,4,23], adj [B,4,4], eps [B,A] or None ->
        dict(logits, value[, action, logp]).  With eps ONE launch (`ddrl_graphnet_act`: forward + DiagGaussian sample),
        without it `ddrl_graphnet_forward`.  A node id outside 0..3 raises (the kernels would clamp it)."""
        B = state.shape[0]
        if tuple(node_idx.shape) != (B,) or node_idx.dtype != torch.int32 or not node_idx.is_cuda:
            raise DDRLError(f"compute_actions: node_idx must be an int32 CUDA tensor of shape {(B,)}")
        if int(((node_idx < 0) | (node_idx > 3)).sum().item()):
            raise DDRLError("compute_actions: node ids must be 0..3 (FL, HL, HR, FR)")
        th = self.theta.reshape(-1)
        if eps is None:
            logits, value = K.graphnet_forward(th, node_idx, state, adj, self.A)
            return {"logits": logits, "value": value}
        logits, value, action, logp = K.graphnet_act(th, node_idx, state, adj, eps, self.A)
        return {"logits": logits, "value": value, "action": action, "logp": logp}

    def learn_on_rollout(self, node_idx, state, adj, boot_node_idx, boot_state, boot_adj, rewards, dones, eps, perms,
                         shuffle=None, cols_per_env: int = 4) -> List[Dict[str, float]]:
        """node_idx [T,C] i32, state [T,C,4,23], adj [T,C,4,4], boot_* the same without T, rewards [T,C],
        dones [T,C/cpe] u8, eps [T,C,A], perms [E,nb] i32, shuffle [T*C] i32 or None."""
        T, Cc = node_idx.shape
        A, cfg, dev, f32 = self.A, self.cfg, self.device, torch.float32
        R = T * Cc
        th = self.theta.reshape(-1)
        idx_f, st_f, adj_f = node_idx.reshape(R), state.reshape(R, 4, 23), adj.reshape(R, 4, 4)
        logits, value = K.graphnet_forward(th, idx_f, st_f, adj_f, A)
        act, logp = K.dg_sample(logits, eps.reshape(R, A).contiguous())
        _, vboot = K.graphnet_forward(th, boot_node_idx.reshape(Cc), boot_state, boot_adj, A)
        adv, vtarg, moments = K.gae(rewards.reshape(1, T, Cc), value.reshape(1, T, Cc), dones, vboot.reshape(1, Cc),
                                    cols_per_env, cfg.gamma, cfg.lambda_)
        if self.world > 1:
            self.dist.all_reduce(moments)
        K.adv_standardize(adv, moments)
        cols = {"idx": idx_f, "st": st_f, "adj": adj_f, "act": act, "logits": logits, "logp": logp,
                "value": value, "adv": adv.reshape(R), "vtarg": vtarg.reshape(R)}
        return self._sgd_phase(cols, perms, shuffle, R)

    def learn_on_batch(self, node_idx, state, adj, actions, action_dist_inputs, action_logp, vf_preds, advantages,
                       value_targets, perms, shuffle=None, standardize: bool = True) -> List[Dict[str, float]]:
        """The learner half only, on POSTPROCESSED sample-batch columns (what RLlib's `Policy.learn_on_batch` receives for the
        shared graph policy): node_idx [R] i32, state [R,4,23], adj [R,4,4] (the observation tuple), actions [R,A],
        action_dist_inputs [R,2A], action_logp / vf_preds / advantages / value_targets [R] — float32 CUDA tensors.
        StandardizeFields -> shuffle -> E x nb minibatch steps -> KL update, as in `learn_on_rollout`."""
        R = state.shape[0]
        adv = advantages.reshape(1, R).clone()
        if standardize:
            self.standardize_advantages(adv)
        cols = {"idx": node_idx.reshape(R), "st": state, "adj": adj, "act": actions, "logits": action_dist_inputs,
                "logp": action_logp, "value": vf_preds, "adv": adv.reshape(R), "vtarg": value_targets}
        for name, t in cols.items():
            want = torch.int32 if name == "idx" else torch.float32
            if t.shape[0] != R or t.dtype != want or not t.is_cuda:
                raise DDRLError(f"learn_on_batch: column {name!r} must be a {want} CUDA tensor with {R} rows, got {t.dtype} "
                                f"{tuple(t.shape)} on {t.device}")
        return self._sgd_phase(cols, perms, shuffle, R)

    def _sgd_phase(self, cols, perms, shuffle, R: int) -> List[Dict[str, float]]:
        """shuffle + E x nb minibatch steps over the prepared columns + stats + KL-coefficient update."""
        A, cfg, dev, f32 = self.A, self.cfg, self.device, torch.float32
        th = self.theta.reshape(-1)
        if shuffle is not None:
            sl = shuffle.long()
            cols = {k: v[sl].contiguous() for k, v in cols.items()}
        MB = min(local_minibatch(cfg.sgd_minibatch_size, self.world), R)
        if MB < 1:
            raise DDRLError("sgd_minibatch_size smaller than the number of ranks")
        E, nb = perms.shape
        if nb != max(1, R // MB):
            raise DDRLError(f"perms has {nb} minibatches per epoch, expected {max(1, R // MB)}")
        hyper = self._hyper(MB * self.world)
        if self.step_kind == "tc":
            return self._sgd_phase_tc(cols, perms, R, MB, E, nb, hyper)
        G = min(self.ctas, MB)
        LG = max(1, min(64, (MB + 255) // 256))
        dlogits = torch.empty(MB, 2 * A, dtype=f32, device=dev)
        dvalue = torch.empty(MB, dtype=f32, device=dev)
        gpart = torch.empty(G, K.part_stride(self.NP), dtype=f32, device=dev)
        spart = torch.empty(1, LG, K.NSTAT, dtype=torch.float64, device=dev)
        step_stats = torch.zeros(E * nb, 1, K.NSTAT, dtype=torch.float64, device=dev)
        ws = None
        if self.two_launch_step:
            spart = torch.empty(1, K.graphnet_train_stat_parts(MB), K.NSTAT, dtype=torch.float64, device=dev)
        order = perms.cpu().numpy()
        self.step_ctr.zero_()
        for e in range(E):
            for i in range(nb):
                r0 = int(order[e, i]) * MB
                sl = slice(r0, r0 + MB)
                if self.two_launch_step:
                    ws = K.graphnet_train_step(th, cols["idx"][sl], cols["st"][sl], cols["adj"][sl], cols["act"][sl],
                                               cols["logits"][sl], cols["logp"][sl], cols["value"][sl], cols["adv"][sl],
                                               cols["vtarg"][sl], A, self.kl_coeff, hyper, G, gpart, spart, ws)
                else:
                    lg, vl = K.graphnet_forward(th, cols["idx"][sl], cols["st"][sl], cols["adj"][sl], A)
                    K.ppo_loss_grad(lg.reshape(1, MB, 2 * A), vl.reshape(1, MB), cols["act"][sl], cols["logits"][sl],
                                    cols["logp"][sl], cols["value"][sl], cols["adv"][sl], cols["vtarg"][sl], A,
                                    self.kl_coeff, hyper, LG, dlogits, dvalue, spart)
                    _lib_backward(th, cols["idx"][sl], cols["st"][sl], cols["adj"][sl], dlogits, dvalue, MB, A, G, gpart)
                # grad_part [G, NP] -> grad [1, NP]; loss-stat partials [1, LG, 8] -> step_stats[step]
                K.grad_reduce(gpart, None, 1, G, self.NP, self.grad)
                _reduce_stats(spart, step_stats, self.step_ctr)
                if self.world > 1:
                    self.dist.all_reduce(self.grad)
                self._adam()
        last = step_stats[E * nb - nb:].clone()
        if self.world > 1:
            self.dist.all_reduce(last)
        stats = finalize_stats(last.cpu().numpy(), self.kl_coeff_host, cfg, MB * self.world)
        self._update_kl(stats)
        return stats


def _graphnet_sgd_phase_tc(self, cols, perms, R: int, MB: int, E: int, nb: int, hyper) -> List[Dict[str, float]]:
    """ONE persistent launch of `ddrl_graphnet_train_step_tc` (all E * nb optimizer steps, fused tail) + stats + KL update."""
    cfg, dev, A = self.cfg, self.device, self.A
    steps = E * nb
    Gn = max(1, min(self.ctas, self.sms // 2))
    key = (steps, Gn)
    if self._tc is None or self._tc["key"] != key:
        self._tc = {"key": key,
                    "mb_perm": torch.empty(steps, dtype=torch.int32, device=dev),
                    "grad_part": torch.empty(Gn, K.part_stride(self.NP), dtype=torch.float32, device=dev),
                    "stat_part": torch.zeros(2 * Gn, K.NSTAT, dtype=torch.float64, device=dev),
                    "step_stats": torch.zeros(steps, 1, K.NSTAT, dtype=torch.float64, device=dev),
                    "tail_bar": torch.zeros(8, dtype=torch.int32, device=dev),
                    "tail_sq": torch.zeros(1, 2 * Gn, 32, dtype=torch.float32, device=dev)}
    w = self._tc
    w["mb_perm"].copy_(perms.reshape(steps))
    self.step_ctr.zero_()
    self.status.zero_()
    if self.world > 1:
        self.dist.all_reduce(self.sync_token)      # line the ranks' streams up ahead of the bounded peer spins
    tail = K.make_sgd_tail(self.theta, self.m, self.v, self.beta_pow, self.grad, w["tail_bar"], w["tail_sq"], cfg.lr, cfg.beta1,
                           cfg.beta2, cfg.adam_eps, cfg.grad_clip, self.gnorm, step_stats=w["step_stats"], step_ctr=self.step_ctr,
                           status=self.status)
    tail.nsteps = steps
    if self.world > 1:
        pkey = (1, self.NP, 2 * Gn)
        if self._peers is None or self._peers.key != pkey:
            from .peer import PeerExchange
            if self._peers is not None:
                self._peers.close()
            self._peers = PeerExchange(self.dist, self.world, self.rank, 1, self.NP, 2 * Gn, dev)
        self._peers.fill(tail)
    th = self.theta.reshape(-1)
    K.graphnet_train_step_tc(th, cols["idx"], cols["st"], cols["adj"], cols["act"], cols["logits"], cols["logp"], cols["value"],
                             cols["adv"], cols["vtarg"], A, MB, w["mb_perm"], self.step_ctr, self.kl_coeff, hyper, Gn,
                             w["grad_part"], w["stat_part"], self.status, tail)      # all E * nb steps in ONE launch
    last = w["step_stats"][steps - nb:].clone()
    if self.world > 1:
        self.dist.all_reduce(last)
    stats = finalize_stats(last.cpu().numpy(), self.kl_coeff_host, cfg, MB * self.world)
    code = int(self.status.item())
    if code:
        what = [n for bit, n in ((1, "MMA completion timed out"), (8, "dl overflow"), (16, "dy overflow"),
                                 (64, "fused-tail barrier / peer wait timed out")) if code & bit]
        raise DDRLError("GraphNet SGD step failed (" + ", ".join(what) + ")" +
                        (" — fp16 split range exceeded: use step='three-kernel' for this workload" if code & 24 else ""))
    self._update_kl(stats)
    return stats


GraphNetLearner._sgd_phase_tc = _graphnet_sgd_phase_tc


def _lib_backward(th, idx, st, adj, dlogits, dvalue, B, A, G, gpart):
    from . import _lib
    f32 = torch.float32
    _lib.check(_lib.load().ddrl_graphnet_backward(K._p(th, f32, "theta"), K._p(idx, torch.int32, "node_idx"),
                                                  K._p(st, f32, "state"), K._p(adj, f32, "adj"),
                                                  K._p(dlogits, f32, "dlogits"), K._p(dvalue, f32, "dvalue"), B, A, G,
                                                  K._p(gpart, f32, "grad_part"), K._stream()), "graphnet_backward")


def _reduce_stats(spart: torch.Tensor, step_stats: torch.Tensor, step_ctr: torch.Tensor):
    """stat partials [1, LG, 8] -> step_stats[*step_ctr] via the C-ABI reducer (its gradient half runs on a dummy)."""
    P, LG, _ = spart.shape
    dummy = _reduce_stats.__dict__.setdefault("dummy", {})
    key = (spart.device, LG)
    if key not in dummy:
        # NP = 1 -> the reducer strides the partial rows by part_stride(1) = 4 floats
        dummy[key] = (torch.zeros(P, LG, K.part_stride(1), dtype=torch.float32, device=spart.device),
                      torch.zeros(P, 1, dtype=torch.float32, device=spart.device))
    gp, g = dummy[key]
    K.grad_reduce(gp, spart, P, LG, 1, g, step_stats, step_ctr)

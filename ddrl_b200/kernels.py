"""Thin torch-tensor wrappers over the C ABI (include/ddrl_b200.h).

PyTorch is plumbing only: device memory, the current CUDA stream, ``torch.distributed``.  Every
function validates device / dtype / contiguity, passes raw pointers to ``libddrl_b200.so`` and raises
``DDRLError`` on any failure — there is no eager/PyTorch fallback."""
from __future__ import annotations

import ctypes as C
from typing import Optional, Tuple

import torch

from . import _lib
from ._lib import DDRLError, PPOHyper, SgdTail

HIDDEN = 64
NSTAT = 8
GN_NODES, GN_FEATS, GN_ENC_IN = 4, 19, 4


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _p(t: Optional[torch.Tensor], dtype=None, name: str = "tensor") -> Optional[int]:
    if t is None:
        return None
    if not t.is_cuda:
        raise DDRLError(f"{name} must be a CUDA tensor (ddrl_b200 has no CPU path)")
    if dtype is not None and t.dtype != dtype:
        raise DDRLError(f"{name} must be {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise DDRLError(f"{name} must be contiguous")
    return t.data_ptr()


def fcnet_num_params(D: int, A: int) -> int:
    n = _lib.load().ddrl_fcnet_num_params(D, A)
    if n < 0:
        raise DDRLError(f"unsupported FCNet shape D={D} A={A}")
    return n


def graphnet_num_params(num_outputs: int) -> int:
    n = _lib.load().ddrl_graphnet_num_params(num_outputs)
    if n < 0:
        raise DDRLError(f"unsupported GraphNet num_outputs={num_outputs}")
    return n


def launch_count() -> int:
    return int(_lib.load().ddrl_launch_count())


# --------------------------------------------------------------------------------------------------
def filter_update(x: torch.Tensor, n: torch.Tensor, M: torch.Tensor, S: torch.Tensor,
                  norm: Optional[torch.Tensor] = None, ws: Optional[torch.Tensor] = None) -> torch.Tensor:
    """x [P,R,D] f32/f64; n [P] i64, M,S [P,D] f64 updated in place; returns norm [P,2,D] f64."""
    lib = _lib.load()
    P, R, D = x.shape
    if norm is None:
        norm = torch.empty(P, 2, D, dtype=torch.float64, device=x.device)
    nbytes = lib.ddrl_filter_ws_bytes(P, R, D)
    if ws is None or ws.numel() * ws.element_size() < nbytes:
        ws = torch.empty(max(nbytes, 8), dtype=torch.uint8, device=x.device)
    if x.dtype not in (torch.float32, torch.float64):
        raise DDRLError("filter_update: x must be float32 or float64")
    _lib.check(lib.ddrl_filter_update(_p(x, None, "x"), int(x.dtype == torch.float64), P, R, D,
                                      _p(n, torch.int64, "n"), _p(M, torch.float64, "M"), _p(S, torch.float64, "S"),
                                      _p(norm, torch.float64, "norm"), _p(ws, None, "ws"), _stream()),
               "filter_update")
    return norm


def fcnet_image_floats(D: int, A: int) -> int:
    return int(_lib.load().ddrl_fcnet_image_floats(D, A))


def fcnet_pack(theta: torch.Tensor, D: int, A: int, img: Optional[torch.Tensor] = None) -> torch.Tensor:
    """theta [P,NP] -> packed shared-memory image [P, image_floats] (see ddrl_b200.h)."""
    P = theta.shape[0]
    if img is None:
        img = torch.empty(P, fcnet_image_floats(D, A), dtype=torch.float32, device=theta.device)
    _lib.check(_lib.load().ddrl_fcnet_pack(_p(theta, torch.float32, "theta"), P, D, A, _p(img, torch.float32, "img"),
                                           _stream()), "fcnet_pack")
    return img


def fcnet_forward(theta: torch.Tensor, obs: torch.Tensor, A: int, norm: Optional[torch.Tensor] = None,
                  clip: float = 0.0, eps: Optional[torch.Tensor] = None, want_obs_out: bool = False,
                  out: Optional[dict] = None, img: Optional[torch.Tensor] = None) -> dict:
    """theta [P,NP], obs [P,R,D] -> dict(logits [P,R,2A], value [P,R], [obs_out], [action, logp])."""
    lib = _lib.load()
    P, R, D = obs.shape
    dev = obs.device
    out = out or {}
    f32 = torch.float32
    logits = out.get("logits") if "logits" in out else torch.empty(P, R, 2 * A, dtype=f32, device=dev)
    value = out.get("value") if "value" in out else torch.empty(P, R, dtype=f32, device=dev)
    obs_out = out.get("obs_out") if "obs_out" in out else (torch.empty_like(obs) if want_obs_out else None)
    action = logp = None
    if eps is not None:
        action = out.get("action") if "action" in out else torch.empty(P, R, A, dtype=f32, device=dev)
        logp = out.get("logp") if "logp" in out else torch.empty(P, R, dtype=f32, device=dev)
    if theta.shape != (P, fcnet_num_params(D, A)):
        raise DDRLError(f"theta shape {tuple(theta.shape)} != ({P}, {fcnet_num_params(D, A)})")
    _lib.check(lib.ddrl_fcnet_forward(_p(theta, f32, "theta"), _p(img, f32, "img"), _p(obs, f32, "obs"),
                                      _p(norm, torch.float64, "norm"),
                                      float(clip), P, R, D, A, _p(obs_out, f32, "obs_out"), _p(logits, f32, "logits"),
                                      _p(value, f32, "value"), _p(eps, f32, "eps"), _p(action, f32, "action"),
                                      _p(logp, f32, "logp"), _stream()), "fcnet_forward")
    res = {"logits": logits, "value": value}
    if obs_out is not None:
        res["obs_out"] = obs_out
    if eps is not None:
        res["action"], res["logp"] = action, logp
    return res


def gae(rewards: torch.Tensor, values: torch.Tensor, dones: torch.Tensor, v_boot: torch.Tensor,
        cols_per_env: int, gamma: float, lam: float, adv: Optional[torch.Tensor] = None,
        vtarg: Optional[torch.Tensor] = None, moments: Optional[torch.Tensor] = None,
        ws: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    """rewards, values [P,T,C] f32; dones [T,C/cols_per_env] u8; v_boot [P,C] -> adv, vtarg, moments [P,3] f64."""
    lib = _lib.load()
    P, T, Cc = rewards.shape
    dev = rewards.device
    adv = adv if adv is not None else torch.empty_like(rewards)
    vtarg = vtarg if vtarg is not None else torch.empty_like(rewards)
    moments = moments if moments is not None else torch.empty(P, 3, dtype=torch.float64, device=dev)
    nbytes = lib.ddrl_gae_ws_bytes(P, Cc)
    if ws is None or ws.numel() * ws.element_size() < nbytes:
        ws = torch.empty(max(nbytes, 8), dtype=torch.uint8, device=dev)
    if tuple(dones.shape) != (T, Cc // cols_per_env):
        raise DDRLError(f"dones shape {tuple(dones.shape)} != ({T}, {Cc // cols_per_env})")
    _lib.check(lib.ddrl_gae(_p(rewards, torch.float32, "rewards"), _p(values, torch.float32, "values"),
                            _p(dones, torch.uint8, "dones"), _p(v_boot, torch.float32, "v_boot"), P, T, Cc,
                            cols_per_env, float(gamma), float(lam), _p(adv, torch.float32, "adv"),
                            _p(vtarg, torch.float32, "vtarg"), _p(moments, torch.float64, "moments"),
                            _p(ws, None, "ws"), _stream()), "gae")
    return adv, vtarg, moments


def adv_standardize(adv: torch.Tensor, moments: torch.Tensor) -> torch.Tensor:
    P = adv.shape[0]
    R = adv.numel() // P
    _lib.check(_lib.load().ddrl_adv_standardize(_p(adv, torch.float32, "adv"), _p(moments, torch.float64, "moments"),
                                                P, R, _stream()), "adv_standardize")
    return adv


def gather_rows(src: torch.Tensor, perm: torch.Tensor, dst: Optional[torch.Tensor] = None) -> torch.Tensor:
    """src [P,R,W] (or [P,R]) f32, perm [P,R] i32 -> dst[p,i] = src[p,perm[p,i]]."""
    P, R = src.shape[:2]
    W = src.numel() // (P * R)
    dst = dst if dst is not None else torch.empty_like(src)
    _lib.check(_lib.load().ddrl_gather_rows(_p(src, torch.float32, "src"), _p(perm, torch.int32, "perm"), P, R, W,
                                            _p(dst, torch.float32, "dst"), _stream()), "gather_rows")
    return dst


def ppo_train_step(theta, obs, actions, old_logits, old_logp, vf_preds, adv, vtarg, A: int, MB: int,
                   mb_perm, step_ctr, kl_coeff, hyper: PPOHyper, ctas_per_policy: int, grad_part, stat_part,
                   ext_dlogits=None, ext_dvalue=None, img=None, tail: Optional[SgdTail] = None):
    lib = _lib.load()
    P, R, D = obs.shape
    f32 = torch.float32
    perm_stride = mb_perm.shape[-1] if mb_perm is not None else 0
    _lib.check(lib.ddrl_ppo_train_step(
        _p(theta, f32, "theta"), _p(img, f32, "img"), _p(obs, f32, "obs"), _p(actions, f32, "actions"),
        _p(old_logits, f32, "old_logits"),
        _p(old_logp, f32, "old_logp"), _p(vf_preds, f32, "vf_preds"), _p(adv, f32, "adv"), _p(vtarg, f32, "vtarg"),
        _p(ext_dlogits, f32, "ext_dlogits"), _p(ext_dvalue, f32, "ext_dvalue"), P, R, D, A, MB,
        _p(mb_perm, torch.int32, "mb_perm"), perm_stride, _p(step_ctr, torch.int32, "step_ctr"),
        _p(kl_coeff, f32, "kl_coeff"), C.byref(hyper) if hyper is not None else None, ctas_per_policy,
        _p(grad_part, f32, "grad_part"), _p(stat_part, torch.float64, "stat_part"),
        C.byref(tail) if tail is not None else None, _stream()), "ppo_train_step")


def grad_reduce(grad_part, stat_part, P: int, G: int, NP: int, grad, step_stats=None, step_ctr=None):
    _lib.check(_lib.load().ddrl_grad_reduce(_p(grad_part, torch.float32, "grad_part"),
                                            _p(stat_part, torch.float64, "stat_part"), P, G, NP,
                                            _p(grad, torch.float32, "grad"), _p(step_stats, torch.float64, "step_stats"),
                                            _p(step_ctr, torch.int32, "step_ctr"), _stream()), "grad_reduce")


def part_stride(NP: int) -> int:
    """Row stride (floats) of the per-CTA gradient partials: NP rounded up to a multiple of 4."""
    return (NP + 3) & ~3


def clip_adam(theta, m, v, beta_pow, grad, lr: float, beta1: float, beta2: float, eps: float, grad_clip: float,
              sync_ws, gnorm_out=None, step_ctr=None, img=None, img_D: int = 0, img_A: int = 0, tc_img=None):
    P, NP = theta.shape
    f32 = torch.float32
    _lib.check(_lib.load().ddrl_clip_adam(_p(theta, f32, "theta"), _p(m, f32, "m"), _p(v, f32, "v"),
                                          _p(beta_pow, f32, "beta_pow"), _p(grad, f32, "grad"), P, NP, float(lr),
                                          float(beta1), float(beta2), float(eps), float(grad_clip),
                                          _p(gnorm_out, f32, "gnorm_out"), _p(step_ctr, torch.int32, "step_ctr"),
                                          _p(sync_ws, torch.int32, "sync_ws"), _p(img, f32, "img"),
                                          _p(tc_img, torch.uint8, "tc_img"), int(img_D), int(img_A), _stream()),
               "clip_adam")


def fcnet_backward(theta, obs, dlogits, dvalue, A: int, ctas_per_policy: Optional[int] = None) -> torch.Tensor:
    """External-gradient backward of the grouped FCNet: -> dtheta [P,NP] (torch.autograd boundary)."""
    P, R, D = obs.shape
    NP = theta.shape[1]
    G = ctas_per_policy or max(1, min((R + 63) // 64, 148 // P))
    gp = torch.empty(P, G, part_stride(NP), dtype=torch.float32, device=obs.device)
    grad = torch.empty(P, NP, dtype=torch.float32, device=obs.device)
    ppo_train_step(theta, obs, None, None, None, None, None, None, A, R, None, None, None, None, G, gp, None,
                   ext_dlogits=dlogits, ext_dvalue=dvalue)
    grad_reduce(gp, None, P, G, NP, grad)
    return grad


# --------------------------------------------------------------------------------------------------
def graphnet_set_variant(variant: int) -> None:
    """Forward schedule of the GraphNet kernels: 0 row-per-CTA, 1 row-per-warp, -1 library default."""
    _lib.check(_lib.load().ddrl_graphnet_set_variant(int(variant)), "graphnet_set_variant")


def graphnet_forward(theta, node_idx, state, adj, A: int, out: Optional[Tuple[torch.Tensor, torch.Tensor]] = None):
    """theta [NP] (actor|critic), node_idx [B] i32, state [B,4,23], adj [B,4,4] -> logits [B,2A], value [B]
    (written into ``out`` = (logits, value) when given)."""
    B = state.shape[0]
    f32 = torch.float32
    if out is not None:
        logits, value = out
        if tuple(logits.shape) != (B, 2 * A) or tuple(value.shape) != (B,):
            raise DDRLError(f"graphnet: out shapes {tuple(logits.shape)} / {tuple(value.shape)} != ({B}, {2 * A}) / ({B},)")
    else:
        logits = torch.empty(B, 2 * A, dtype=f32, device=state.device)
        value = torch.empty(B, dtype=f32, device=state.device)
    if tuple(state.shape[1:]) != (GN_NODES, GN_FEATS + GN_ENC_IN) or tuple(adj.shape[1:]) != (GN_NODES, GN_NODES):
        raise DDRLError(f"graphnet: state {tuple(state.shape)} / adj {tuple(adj.shape)} must be [B,4,23] / [B,4,4]")
    if theta.numel() != graphnet_num_params(2 * A):
        raise DDRLError(f"graphnet: theta has {theta.numel()} params, expected {graphnet_num_params(2 * A)}")
    _lib.check(_lib.load().ddrl_graphnet_forward(_p(theta, f32, "theta"), _p(node_idx, torch.int32, "node_idx"),
                                                 _p(state, f32, "state"), _p(adj, f32, "adj"), B, A,
                                                 _p(logits, f32, "logits"), _p(value, f32, "value"), _stream()),
               "graphnet_forward")
    return logits, value


def graphnet_act(theta, node_idx, state, adj, eps, A: int, out: Optional[Tuple[torch.Tensor, ...]] = None):
    """GraphNet forward + DiagGaussian sample in ONE launch: theta [NP], node_idx [B] i32, state [B,4,23], adj [B,4,4],
    eps [B,A] -> logits [B,2A], value [B], action [B,A], logp [B] (written into ``out`` = (logits, value, action, logp) when
    given).  Bit-identical to ``graphnet_forward`` under forward variant 1 followed by ``dg_sample``."""
    B = state.shape[0]
    f32 = torch.float32
    shapes = ((B, 2 * A), (B,), (B, A), (B,))
    if out is not None:
        if len(out) != 4 or any(tuple(t.shape) != s for t, s in zip(out, shapes)):
            raise DDRLError(f"graphnet_act: out shapes {[tuple(t.shape) for t in out]} != {list(shapes)}")
        logits, value, action, logp = out
    else:
        logits, value, action, logp = (torch.empty(s, dtype=f32, device=state.device) for s in shapes)
    if tuple(state.shape[1:]) != (GN_NODES, GN_FEATS + GN_ENC_IN) or tuple(adj.shape[1:]) != (GN_NODES, GN_NODES):
        raise DDRLError(f"graphnet: state {tuple(state.shape)} / adj {tuple(adj.shape)} must be [B,4,23] / [B,4,4]")
    if tuple(eps.shape) != (B, A):
        raise DDRLError(f"graphnet_act: eps {tuple(eps.shape)} must be [{B}, {A}]")
    if theta.numel() != graphnet_num_params(2 * A):
        raise DDRLError(f"graphnet: theta has {theta.numel()} params, expected {graphnet_num_params(2 * A)}")
    _lib.check(_lib.load().ddrl_graphnet_act(_p(theta, f32, "theta"), _p(node_idx, torch.int32, "node_idx"),
                                             _p(state, f32, "state"), _p(adj, f32, "adj"), _p(eps, f32, "eps"), B, A,
                                             _p(logits, f32, "logits"), _p(value, f32, "value"), _p(action, f32, "action"),
                                             _p(logp, f32, "logp"), _stream()), "graphnet_act")
    return logits, value, action, logp


def graphnet_backward(theta, node_idx, state, adj, dlogits, dvalue, A: int, ctas: Optional[int] = None):
    B = state.shape[0]
    f32 = torch.float32
    NP = theta.numel()
    G = ctas or max(1, min(B, 74))
    gp = torch.zeros(G, part_stride(NP), dtype=f32, device=state.device)
    grad = torch.empty(1, NP, dtype=f32, device=state.device)
    _lib.check(_lib.load().ddrl_graphnet_backward(_p(theta, f32, "theta"), _p(node_idx, torch.int32, "node_idx"),
                                                  _p(state, f32, "state"), _p(adj, f32, "adj"),
                                                  _p(dlogits, f32, "dlogits"), _p(dvalue, f32, "dvalue"), B, A, G,
                                                  _p(gp, f32, "grad_part"), _stream()), "graphnet_backward")
    grad_reduce(gp, None, 1, G, NP, grad)
    return grad.reshape(-1)


def gcn_forward(x, adj, W, b=None, act: str = "tanh"):
    B, n, F = x.shape
    U = W.shape[1]
    y = torch.empty(B, n, U, dtype=torch.float32, device=x.device)
    f32 = torch.float32
    _lib.check(_lib.load().ddrl_gcn_forward(_p(x, f32, "x"), _p(adj, f32, "adj"), _p(W, f32, "W"), _p(b, f32, "b"), B,
                                            F, U, {"tanh": 1, None: 0, "linear": 0}[act], _p(y, f32, "y"), _stream()),
               "gcn_forward")
    return y


_ACT = {"tanh": 1, None: 0, "linear": 0}


def mpnn2_forward(x, adj, W_msg, W_upd, b=None, act: str = "tanh"):
    """MPNN2 (models/gcn.py:96-150): x [B,4,F], adj [B,4,4], W_msg [2F,U], W_upd [F+U,U] -> [B,4,U]."""
    B, n, F = x.shape
    U = W_upd.shape[1]
    if n != 4 or tuple(W_msg.shape) != (2 * F, U) or tuple(W_upd.shape) != (F + U, U):
        raise DDRLError(f"mpnn2_forward: bad shapes x {tuple(x.shape)} W_msg {tuple(W_msg.shape)} W_upd {tuple(W_upd.shape)}")
    y = torch.empty(B, n, U, dtype=torch.float32, device=x.device)
    f32 = torch.float32
    _lib.check(_lib.load().ddrl_mpnn2_forward(_p(x, f32, "x"), _p(adj, f32, "adj"), _p(W_msg, f32, "W_msg"), _p(W_upd, f32, "W_upd"),
                                              _p(b, f32, "b"), B, F, U, _ACT[act], _p(y, f32, "y"), _stream()), "mpnn2_forward")
    return y


def _graph_layer_backward(fn_name, x, adj, W0, W1, b, dy, NPw: int, act: str, ctas: Optional[int], need_dx: bool):
    B, n, F = x.shape
    U = dy.shape[2]
    f32 = torch.float32
    G = ctas or int(max(1, min(B, 148 * 2)))
    gp = torch.empty(G, part_stride(NPw), dtype=f32, device=x.device)
    dx = torch.empty(B, n, F, dtype=f32, device=x.device) if need_dx else None
    fn = getattr(_lib.load(), fn_name)
    _lib.check(fn(_p(x, f32, "x"), _p(adj, f32, "adj"), _p(W0, f32, "W0"), _p(W1, f32, "W1"), _p(b, f32, "b"), _p(dy, f32, "dy"),
                  B, F, U, _ACT[act], G, _p(dx, f32, "dx"), _p(gp, f32, "grad_part"), _stream()), fn_name)
    g = torch.empty(1, NPw, dtype=f32, device=x.device)
    grad_reduce(gp, None, 1, G, NPw, g)
    return dx, g.reshape(-1)


def mpnn2_backward(x, adj, W_msg, W_upd, b, dy, act: str = "tanh", ctas: Optional[int] = None, need_dx: bool = True):
    """Backward of MPNN2: dy [B,4,U] -> (dx [B,4,F] or None, dW_msg [2F,U], dW_upd [F+U,U], db [U])."""
    B, n, F = x.shape
    U = W_upd.shape[1]
    if n != 4 or tuple(W_msg.shape) != (2 * F, U) or tuple(W_upd.shape) != (F + U, U) or tuple(dy.shape) != (B, n, U):
        raise DDRLError("mpnn2_backward: bad shapes")
    dx, g = _graph_layer_backward("ddrl_mpnn2_backward", x, adj, W_msg, W_upd, b, dy, 2 * F * U + (F + U) * U + U, act, ctas, need_dx)
    o1, o2 = 2 * F * U, 2 * F * U + (F + U) * U
    return dx, g[:o1].reshape(2 * F, U), g[o1:o2].reshape(F + U, U), g[o2:]


def gat1_backward(x, adj, W_pre, w_att, b, dy, act: str = "tanh", ctas: Optional[int] = None, need_dx: bool = True):
    """Backward of GAT1: dy [B,4,U] -> (dx [B,4,F] or None, dW_pre [F,U], dw_att [2U], db [U])."""
    B, n, F = x.shape
    U = W_pre.shape[1]
    w_att = w_att.reshape(-1).contiguous()
    if n != 4 or W_pre.shape[0] != F or w_att.numel() != 2 * U or tuple(dy.shape) != (B, n, U):
        raise DDRLError("gat1_backward: bad shapes")
    dx, g = _graph_layer_backward("ddrl_gat1_backward", x, adj, W_pre, w_att, b, dy, F * U + 3 * U, act, ctas, need_dx)
    return dx, g[:F * U].reshape(F, U), g[F * U:F * U + 2 * U], g[F * U + 2 * U:]


def gat1_forward(x, adj, W_pre, w_att, b=None, act: str = "tanh"):
    """GAT1 (models/gcn.py:153-206): x [B,4,F], adj [B,4,4], W_pre [F,U], w_att [2U] (or [2U,1]) -> [B,4,U]."""
    B, n, F = x.shape
    U = W_pre.shape[1]
    w_att = w_att.reshape(-1)
    if n != 4 or W_pre.shape[0] != F or w_att.numel() != 2 * U:
        raise DDRLError(f"gat1_forward: bad shapes x {tuple(x.shape)} W_pre {tuple(W_pre.shape)} w_att {tuple(w_att.shape)}")
    y = torch.empty(B, n, U, dtype=torch.float32, device=x.device)
    f32 = torch.float32
    _lib.check(_lib.load().ddrl_gat1_forward(_p(x, f32, "x"), _p(adj, f32, "adj"), _p(W_pre, f32, "W_pre"), _p(w_att, f32, "w_att"),
                                             _p(b, f32, "b"), B, F, U, _ACT[act], _p(y, f32, "y"), _stream()), "gat1_forward")
    return y


def symm_norm(adj):
    """graph_ops.symm_norm (models/graph_ops.py:3-11): D^-1/2 A D^-1/2, adj [B,N,N]."""
    B, N, _ = adj.shape
    out = torch.empty_like(adj)
    _lib.check(_lib.load().ddrl_symm_norm(_p(adj, torch.float32, "adj"), B, N, _p(out, torch.float32, "out"), _stream()), "symm_norm")
    return out


def segment_softmax(data, segment_ids, num_segments: int):
    """graph_ops.segment_softmax (models/graph_ops.py:23-26): data [E] or [E,C], segment_ids [E] int32."""
    d2 = data.reshape(data.shape[0], -1).contiguous()
    E, Cc = d2.shape
    sums = torch.empty(num_segments, Cc, dtype=torch.float32, device=data.device)
    bad = torch.zeros(1, dtype=torch.int32, device=data.device)
    out = torch.empty_like(d2)
    _lib.check(_lib.load().ddrl_segment_softmax(_p(d2, torch.float32, "data"), _p(segment_ids, torch.int32, "segment_ids"), E, Cc,
                                                int(num_segments), _p(sums, torch.float32, "sums"), _p(bad, torch.int32, "bad"),
                                                _p(out, torch.float32, "out"), _stream()), "segment_softmax")
    if int(bad.item()):
        raise DDRLError("segment_softmax: a segment id is outside [0, num_segments)")
    return out.reshape(data.shape)


def leg_coupling_(logits, node_id, coupling):
    B, W = logits.shape
    f32 = torch.float32
    _lib.check(_lib.load().ddrl_leg_coupling(_p(logits, f32, "logits"), _p(node_id, torch.int32, "node_id"),
                                             _p(coupling, f32, "coupling"), B, W, _stream()), "leg_coupling")
    return logits


def param_expand(theta_model, layout_map, theta_kernel):
    """theta_kernel [P,NPk] = index-select of theta_model [P,NPm] through layout_map [NPk] i32 (>= NPm: constant zero)."""
    P, NPm = theta_model.shape
    NPk = theta_kernel.shape[1]
    _lib.check(_lib.load().ddrl_param_expand(_p(theta_model, torch.float32, "theta_model"), _p(layout_map, torch.int32, "map"), P,
                                             NPm, NPk, _p(theta_kernel, torch.float32, "theta_kernel"), _stream()), "param_expand")
    return theta_kernel


def grad_tie(grad_kernel, inverse_map, grad_model):
    """grad_model [P,NPm] = sum over the (<= 2) kernel-layout copies of every model variable (inverse_map [NPm,2] i32)."""
    P, NPk = grad_kernel.shape
    NPm = grad_model.shape[1]
    _lib.check(_lib.load().ddrl_grad_tie(_p(grad_kernel, torch.float32, "grad_kernel"), _p(inverse_map, torch.int32, "inv"), P,
                                         NPm, NPk, _p(grad_model, torch.float32, "grad_model"), _stream()), "grad_tie")
    return grad_model


def leg_coupling_backward_(dout, logits_pre, node_id, coupling):
    """In place: dout [B,W] becomes the gradient w.r.t. the pre-coupling logits; returns dcoupling [4,2] (see
    ddrl_leg_coupling_backward)."""
    B, W = dout.shape
    f32 = torch.float32
    dc = torch.empty(4, 2, dtype=f32, device=dout.device)
    _lib.check(_lib.load().ddrl_leg_coupling_backward(_p(dout, f32, "dout"), _p(logits_pre, f32, "logits_pre"),
                                                      _p(node_id, torch.int32, "node_id"), _p(coupling, f32, "coupling"), B, W,
                                                      _p(dc, f32, "dcoupling"), _stream()), "leg_coupling_backward")
    return dc


def filter_partial(x: torch.Tensor, ws: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Per-rank half of the filter update: x [P,R,D] -> partials [P, nparts, D, 3] f64 {count, mean, M2}."""
    lib = _lib.load()
    P, R, D = x.shape
    nparts = lib.ddrl_filter_num_partials(R)
    if ws is None:
        ws = torch.empty(P, nparts, D, 3, dtype=torch.float64, device=x.device)
    _lib.check(lib.ddrl_filter_partial(_p(x, None, "x"), int(x.dtype == torch.float64), P, R, D,
                                       _p(ws, torch.float64, "ws"), _stream()), "filter_partial")
    return ws


def filter_merge(parts: torch.Tensor, R_total: int, n, M, S, norm: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Fold parts [P, nparts, D, 3] (fixed order) into the running state; returns norm [P,2,D]."""
    P, nparts, D, _ = parts.shape
    if norm is None:
        norm = torch.empty(P, 2, D, dtype=torch.float64, device=parts.device)
    _lib.check(_lib.load().ddrl_filter_merge(_p(parts, torch.float64, "parts"), nparts, P, D, int(R_total),
                                             _p(n, torch.int64, "n"), _p(M, torch.float64, "M"),
                                             _p(S, torch.float64, "S"), _p(norm, torch.float64, "norm"), _stream()),
               "filter_merge")
    return norm


def filter_stream_ws_bytes(P: int, T: int, C: int, W: int, D: int) -> int:
    n = int(_lib.load().ddrl_filter_stream_ws_bytes(P, T, C, W, D))
    if n < 0:
        raise DDRLError(f"filter_stream: bad shape P={P} T={T} C={C} W={W} D={D} (C must be a multiple of W)")
    return n


def filter_stream(x: torch.Tensor, n: torch.Tensor, M: torch.Tensor, S: torch.Tensor, T: int, W: int, clip: float = 0.0,
                  out: Optional[torch.Tensor] = None, parts: Optional[torch.Tensor] = None,
                  ws: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Row-by-row MeanStdFilter streams (ddrl_filter_stream): x [P,R,D] f32/f64 with R = T*C rows in (t, c) order, W
    streams per policy over equal column blocks, all starting from the running state n [P] i64, M,S [P,D] f64 (read only).
    -> (out [P,R,D] f32 normalised rows, parts [P,W,D,3] f64 {count, mean, M2} of every stream); fold parts into the state
    with `filter_merge(parts, R, n, M, S, norm)`."""
    if x.dtype not in (torch.float32, torch.float64):
        raise DDRLError("filter_stream: x must be float32 or float64")
    P, R, D = x.shape
    if T < 1 or R % T:
        raise DDRLError(f"filter_stream: R={R} rows are not T={T} steps of whole rows")
    C = R // T
    lib = _lib.load()
    nbytes = filter_stream_ws_bytes(P, T, C, W, D)
    if out is None:
        out = torch.empty(P, R, D, dtype=torch.float32, device=x.device)
    if parts is None:
        parts = torch.empty(P, W, D, 3, dtype=torch.float64, device=x.device)
    if ws is None or ws.numel() * ws.element_size() < nbytes:
        ws = torch.empty(max(nbytes, 8), dtype=torch.uint8, device=x.device)
    if tuple(out.shape) != (P, R, D) or tuple(parts.shape) != (P, W, D, 3):
        raise DDRLError(f"filter_stream: out must be {(P, R, D)} and parts {(P, W, D, 3)}")
    _lib.check(lib.ddrl_filter_stream(_p(x, None, "x"), int(x.dtype == torch.float64), P, int(T), int(C), int(W), D,
                                      _p(n, torch.int64, "n"), _p(M, torch.float64, "M"), _p(S, torch.float64, "S"),
                                      float(clip), _p(out, torch.float32, "out"), _p(parts, torch.float64, "parts"),
                                      _p(ws, None, "ws"), _stream()), "filter_stream")
    return out, parts


def ppo_loss_grad(logits, value, actions, old_logits, old_logp, vf_preds, adv, vtarg, A: int, kl_coeff,
                  hyper: PPOHyper, ctas: int, dlogits, dvalue, stat_part):
    """logits [P,R,2A], value [P,R] -> dlogits, dvalue (in the given buffers), stat_part [P,ctas,8] f64."""
    P, R = value.shape
    f32 = torch.float32
    _lib.check(_lib.load().ddrl_ppo_loss_grad(
        _p(logits, f32, "logits"), _p(value, f32, "value"), _p(actions, f32, "actions"),
        _p(old_logits, f32, "old_logits"), _p(old_logp, f32, "old_logp"), _p(vf_preds, f32, "vf_preds"),
        _p(adv, f32, "adv"), _p(vtarg, f32, "vtarg"), P, R, A, _p(kl_coeff, f32, "kl_coeff"), C.byref(hyper), ctas,
        _p(dlogits, f32, "dlogits"), _p(dvalue, f32, "dvalue"), _p(stat_part, torch.float64, "stat_part"), _stream()),
        "ppo_loss_grad")


def graphnet_train_stat_parts(B: int) -> int:
    n = _lib.load().ddrl_graphnet_train_stat_parts(int(B))
    if n < 0:
        raise DDRLError(f"graphnet_train_stat_parts: bad B={B}")
    return n


def graphnet_train_step(theta, node_idx, state, adj, actions, old_logits, old_logp, vf_preds, adv, vtarg, A: int, kl_coeff,
                        hyper: PPOHyper, ctas: int, grad_part, stat_part, ws: Optional[torch.Tensor] = None):
    """One GraphNet SGD step in two launches (forward + PPO loss + backward to the layer inputs per row, then the weight
    gradients): theta [NP], node_idx [B] i32, state [B,4,23], adj [B,4,4], actions [B,A], old_logits [B,2A],
    old_logp / vf_preds / adv / vtarg [B] -> grad_part [ctas, NPs] f32, stat_part [graphnet_train_stat_parts(B), 8] f64.
    ``ws``: uint8 workspace of ddrl_graphnet_train_ws_bytes(B) bytes (allocated when None).  Returns ws for reuse."""
    lib = _lib.load()
    B = state.shape[0]
    f32 = torch.float32
    if tuple(state.shape[1:]) != (GN_NODES, GN_FEATS + GN_ENC_IN) or tuple(adj.shape[1:]) != (GN_NODES, GN_NODES):
        raise DDRLError(f"graphnet: state {tuple(state.shape)} / adj {tuple(adj.shape)} must be [B,4,23] / [B,4,4]")
    if theta.numel() != graphnet_num_params(2 * A):
        raise DDRLError(f"graphnet: theta has {theta.numel()} params, expected {graphnet_num_params(2 * A)}")
    nbytes = int(lib.ddrl_graphnet_train_ws_bytes(B))
    if ws is None or ws.numel() * ws.element_size() < nbytes:
        ws = torch.empty(max(nbytes, 8), dtype=torch.uint8, device=state.device)
    parts = graphnet_train_stat_parts(B)
    if stat_part.numel() != parts * NSTAT or tuple(grad_part.shape) != (ctas, part_stride(theta.numel())):
        raise DDRLError(f"graphnet_train_step: stat_part needs {parts} x {NSTAT} float64, grad_part [{ctas}, "
                        f"{part_stride(theta.numel())}] float32")
    _lib.check(lib.ddrl_graphnet_train_step(
        _p(theta, f32, "theta"), _p(node_idx, torch.int32, "node_idx"), _p(state, f32, "state"), _p(adj, f32, "adj"),
        _p(actions, f32, "actions"), _p(old_logits, f32, "old_logits"), _p(old_logp, f32, "old_logp"),
        _p(vf_preds, f32, "vf_preds"), _p(adv, f32, "adv"), _p(vtarg, f32, "vtarg"), B, A, _p(kl_coeff, f32, "kl_coeff"),
        C.byref(hyper), int(ctas), _p(ws, None, "ws"), _p(grad_part, f32, "grad_part"),
        _p(stat_part, torch.float64, "stat_part"), _stream()), "graphnet_train_step")
    return ws


def graphnet_train_step_tc(theta, node_idx, state, adj, actions, old_logits, old_logp, vf_preds, adv, vtarg, A: int, MB: int,
                           mb_perm, step_ctr, kl_coeff, hyper: PPOHyper, ctas_per_net: int, grad_part, stat_part, status=None,
                           tail: Optional[SgdTail] = None):
    """Persistent tensor-core GraphNet SGD step(s) over ALL R rows of the (shuffled) train batch: theta [NP], node_idx [R] i32,
    state [R,4,23], adj [R,4,4], actions [R,A], old_logits [R,2A], old_logp / vf_preds / adv / vtarg [R]; step k of the launch
    trains minibatch mb_perm[step_ctr + k] (see ddrl_graphnet_train_step_tc).  grad_part [ctas_per_net, NPs] f32, stat_part
    [2 * ctas_per_net, 8] f64 zero-initialised."""
    R = state.shape[0]
    f32 = torch.float32
    if tuple(state.shape[1:]) != (GN_NODES, GN_FEATS + GN_ENC_IN) or tuple(adj.shape[1:]) != (GN_NODES, GN_NODES):
        raise DDRLError(f"graphnet: state {tuple(state.shape)} / adj {tuple(adj.shape)} must be [R,4,23] / [R,4,4]")
    if theta.numel() != graphnet_num_params(2 * A):
        raise DDRLError(f"graphnet: theta has {theta.numel()} params, expected {graphnet_num_params(2 * A)}")
    if tuple(grad_part.shape) != (ctas_per_net, part_stride(theta.numel())) or stat_part.numel() != 2 * ctas_per_net * NSTAT:
        raise DDRLError(f"graphnet_train_step_tc: grad_part must be [{ctas_per_net}, {part_stride(theta.numel())}] f32, stat_part "
                        f"[{2 * ctas_per_net}, {NSTAT}] f64")
    _lib.check(_lib.load().ddrl_graphnet_train_step_tc(
        _p(theta, f32, "theta"), _p(node_idx, torch.int32, "node_idx"), _p(state, f32, "state"), _p(adj, f32, "adj"),
        _p(actions, f32, "actions"), _p(old_logits, f32, "old_logits"), _p(old_logp, f32, "old_logp"),
        _p(vf_preds, f32, "vf_preds"), _p(adv, f32, "adv"), _p(vtarg, f32, "vtarg"), R, A, int(MB),
        _p(mb_perm, torch.int32, "mb_perm"), _p(step_ctr, torch.int32, "step_ctr"), _p(kl_coeff, f32, "kl_coeff"),
        C.byref(hyper), int(ctas_per_net), _p(grad_part, f32, "grad_part"), _p(stat_part, torch.float64, "stat_part"),
        _p(status, torch.int32, "status"), C.byref(tail) if tail is not None else None, _stream()), "graphnet_train_step_tc")


def dg_sample(logits: torch.Tensor, eps: torch.Tensor):
    """logits [R,2A], eps [R,A] -> action [R,A], logp [R]  (DiagGaussian sample, unclipped)."""
    R, A = eps.shape
    f32 = torch.float32
    action = torch.empty(R, A, dtype=f32, device=logits.device)
    logp = torch.empty(R, dtype=f32, device=logits.device)
    _lib.check(_lib.load().ddrl_dg_sample(_p(logits, f32, "logits"), _p(eps, f32, "eps"), R, A, _p(action, f32, "action"),
                                          _p(logp, f32, "logp"), _stream()), "dg_sample")
    return action, logp


def umma_selftest(A: torch.Tensor, B: torch.Tensor, N: int, Kdim: int, a_mn: bool, b_mn: bool, split: bool, M: int = 128):
    """Diagnostic tcgen05 GEMM (see ddrl_b200.h): returns (D [128,N] float32 = raw TMEM lanes, status int)."""
    D = torch.zeros(128, N, dtype=torch.float32, device=A.device)
    status = torch.full((1,), -1, dtype=torch.int32, device=A.device)
    _lib.check(_lib.load().ddrl_umma_selftest(_p(A, torch.float32, "A"), A.shape[0], A.shape[1], _p(B, torch.float32, "B"),
                                              B.shape[0], B.shape[1], M, N, Kdim, int(a_mn), int(b_mn), int(split),
                                              _p(D, torch.float32, "D"), _p(status, torch.int32, "status"), _stream()),
               "umma_selftest")
    return D, int(status.item())


def fcnet_tc_pack(theta: torch.Tensor, D: int, A: int, img: Optional[torch.Tensor] = None) -> torch.Tensor:
    """theta [P,NP] -> tensor-core weight image [P, tc_image_bytes] uint8 (fp16 hi/lo weights + fp32 biases/heads)."""
    lib = _lib.load()
    P = theta.shape[0]
    nbytes = lib.ddrl_fcnet_tc_image_bytes(D, A)
    if nbytes < 0:
        raise DDRLError(f"tensor-core path does not support D={D} A={A}")
    if img is None:
        img = torch.empty(P, nbytes, dtype=torch.uint8, device=theta.device)
    _lib.check(lib.ddrl_fcnet_tc_pack(_p(theta, torch.float32, "theta"), P, D, A, _p(img, torch.uint8, "tc_img"), _stream()),
               "fcnet_tc_pack")
    return img


def fcnet_forward_tc(tc_img, obs, A: int, norm=None, clip: float = 0.0, eps=None, out: Optional[dict] = None,
                     status: Optional[torch.Tensor] = None) -> dict:
    """Inference on the tensor cores (ddrl_fcnet_forward_tc): obs [P,R,D] f32 + tensor-core weight image -> dict(logits,
    value[, obs_out][, action, logp]).  ``out`` may carry preallocated tensors; a None entry skips that output."""
    P, R, D = obs.shape
    f32 = torch.float32
    o = _forward_outputs(obs, A, eps, out, want_obs_out=norm is not None, samples_only=out is not None)
    if status is None:
        status = torch.zeros(1, dtype=torch.int32, device=obs.device)
    _lib.check(_lib.load().ddrl_fcnet_forward_tc(
        _p(tc_img, torch.uint8, "tc_img"), _p(obs, f32, "obs"), _p(norm, torch.float64, "norm"), float(clip or 0.0), P, R, D, A,
        _p(o.get("obs_out"), f32, "obs_out"), _p(o.get("logits"), f32, "logits"), _p(o.get("value"), f32, "value"),
        _p(eps, f32, "eps"), _p(o.get("action"), f32, "action"), _p(o.get("logp"), f32, "logp"),
        _p(status, torch.int32, "status"), _stream()), "fcnet_forward_tc")
    o["status"] = status
    return o


def _forward_outputs(obs, A: int, eps, out: Optional[dict], want_obs_out: bool, samples_only: bool = False) -> dict:
    """Outputs of a forward wrapper: the entries of ``out`` (None skips that output) and a new float32 tensor for each missing
    one (obs_out only if ``want_obs_out``; with ``samples_only`` only action / logp, and those only when eps is given)."""
    P, R, D = obs.shape
    o = dict(out) if out is not None else {}
    shapes = {} if samples_only else {"logits": (P, R, 2 * A), "value": (P, R), "obs_out": (P, R, D) if want_obs_out else None}
    if eps is not None:
        shapes.update(action=(P, R, A), logp=(P, R))
    for k, shp in shapes.items():
        if k not in o:
            o[k] = torch.empty(shp, dtype=torch.float32, device=obs.device) if shp is not None else None
    return o


def fcnet_forward_coupled(theta, obs, node_id, coupling, A: int = 2, norm=None, clip: float = 0.0, eps=None,
                          status: Optional[torch.Tensor] = None, out: Optional[dict] = None, img=None,
                          want_obs_out: bool = False) -> dict:
    """Leg-coupled inference in ONE launch (ddrl_fcnet_forward_coupled, FP32): theta [1,NP] (or the packed image img),
    obs [1,R,D], node_id [1,R] int32 0..3, coupling [4,2] (or the flat 8 entries) -> dict(logits (coupled), value
    [, obs_out][, action, logp], status).  Bit-identical to fcnet_forward -> leg_coupling_ -> dg_sample.  A node id outside
    0..3 sets STATUS_BAD_NODE in ``status`` (a new zeroed int32 [1] unless given); ``out`` entries set to None are skipped."""
    P, R, D = obs.shape
    f32 = torch.float32
    o = _forward_outputs(obs, A, eps, out, want_obs_out)
    if status is None:
        status = torch.zeros(1, dtype=torch.int32, device=obs.device)
    _lib.check(_lib.load().ddrl_fcnet_forward_coupled(
        _p(theta, f32, "theta"), _p(img, f32, "img"), _p(node_id, torch.int32, "node_id"), _p(coupling, f32, "coupling"),
        _p(obs, f32, "obs"), _p(norm, torch.float64, "norm"), float(clip or 0.0), P, R, D, A,
        _p(o.get("obs_out"), f32, "obs_out"), _p(o.get("logits"), f32, "logits"), _p(o.get("value"), f32, "value"),
        _p(eps, f32, "eps"), _p(o.get("action"), f32, "action"), _p(o.get("logp"), f32, "logp"),
        _p(status, torch.int32, "status"), _stream()), "fcnet_forward_coupled")
    o["status"] = status
    return o


def fcnet_forward_tc_coupled(tc_img, obs, node_id, coupling, A: int = 2, norm=None, clip: float = 0.0, eps=None,
                             status: Optional[torch.Tensor] = None, out: Optional[dict] = None,
                             want_obs_out: bool = False) -> dict:
    """Leg-coupled inference on the tensor cores in ONE launch (ddrl_fcnet_forward_tc_coupled; D in {19, 20}): as
    fcnet_forward_coupled with the tensor-core weight image.  Bit-identical to fcnet_forward_tc -> leg_coupling_ -> dg_sample."""
    P, R, D = obs.shape
    f32 = torch.float32
    o = _forward_outputs(obs, A, eps, out, want_obs_out)
    if status is None:
        status = torch.zeros(1, dtype=torch.int32, device=obs.device)
    _lib.check(_lib.load().ddrl_fcnet_forward_tc_coupled(
        _p(tc_img, torch.uint8, "tc_img"), _p(node_id, torch.int32, "node_id"), _p(coupling, f32, "coupling"),
        _p(obs, f32, "obs"), _p(norm, torch.float64, "norm"), float(clip or 0.0), P, R, D, A,
        _p(o.get("obs_out"), f32, "obs_out"), _p(o.get("logits"), f32, "logits"), _p(o.get("value"), f32, "value"),
        _p(eps, f32, "eps"), _p(o.get("action"), f32, "action"), _p(o.get("logp"), f32, "logp"),
        _p(status, torch.int32, "status"), _stream()), "fcnet_forward_tc_coupled")
    o["status"] = status
    return o


def tc_set_variant(variant: int) -> None:
    """0 = automatic (ping-pong kernel when D <= 47), 1 = branch-sequential kernel, 2 = ping-pong kernel (D <= 47)."""
    _lib.check(_lib.load().ddrl_tc_set_variant(int(variant)), "tc_set_variant")


def tc_set_cluster(size: int) -> None:
    """-1 = automatic, 1 = off, 2/4/8/16 = forced thread-block cluster size of the ping-pong kernel."""
    _lib.check(_lib.load().ddrl_tc_set_cluster(int(size)), "tc_set_cluster")


def tc_last_cluster() -> int:
    return int(_lib.load().ddrl_tc_last_cluster())


def tc_pingpong_eligible(D: int, A: int) -> bool:
    return bool(_lib.load().ddrl_tc_pingpong_eligible(int(D), int(A)))


def _step_args(obs, actions, old_logits, old_logp, vf_preds, adv, vtarg, A: int, MB: int, mb_perm, step_ctr, kl_coeff,
               hyper: PPOHyper, ctas_per_policy: int, grad_part, stat_part) -> list:
    """The arguments obs ... stat_part that ddrl_ppo_train_step_tc, _tc_coupled and ddrl_ppo_train_step_coupled share."""
    P, R, D = obs.shape
    f32 = torch.float32
    perm_stride = mb_perm.shape[-1] if mb_perm is not None else 0
    return [_p(obs, f32, "obs"), _p(actions, f32, "actions"), _p(old_logits, f32, "old_logits"), _p(old_logp, f32, "old_logp"),
            _p(vf_preds, f32, "vf_preds"), _p(adv, f32, "adv"), _p(vtarg, f32, "vtarg"), P, R, D, A, MB,
            _p(mb_perm, torch.int32, "mb_perm"), perm_stride, _p(step_ctr, torch.int32, "step_ctr"),
            _p(kl_coeff, f32, "kl_coeff"), C.byref(hyper), ctas_per_policy, _p(grad_part, f32, "grad_part"),
            _p(stat_part, torch.float64, "stat_part")]


def ppo_train_step_tc(tc_img, obs, actions, old_logits, old_logp, vf_preds, adv, vtarg, A: int, MB: int, mb_perm, step_ctr,
                      kl_coeff, hyper: PPOHyper, ctas_per_policy: int, grad_part, stat_part, status=None,
                      tail: Optional[SgdTail] = None):
    _lib.check(_lib.load().ddrl_ppo_train_step_tc(
        _p(tc_img, torch.uint8, "tc_img"),
        *_step_args(obs, actions, old_logits, old_logp, vf_preds, adv, vtarg, A, MB, mb_perm, step_ctr, kl_coeff, hyper,
                    ctas_per_policy, grad_part, stat_part),
        _p(status, torch.int32, "status"), C.byref(tail) if tail is not None else None, _stream()), "ppo_train_step_tc")


STATUS_BAD_NODE = 128      # DDRL_STATUS_BAD_NODE: a node id outside 0..3 reached a leg-coupled step


def ppo_train_step_tc_coupled(tc_img, theta, node_id, obs, actions, old_logits, old_logp, vf_preds, adv, vtarg, A: int, MB: int,
                              mb_perm, step_ctr, kl_coeff, hyper: PPOHyper, ctas_per_policy: int, grad_part, stat_part,
                              status, tail: SgdTail):
    """Leg-coupled tensor-core step (SharedDecentralLegID, ddrl_ppo_train_step_tc_coupled): theta [1, NP + 8] (FCNet
    variables, then leg_coupling [4, 2]), node_id [1, R] int32, grad_part [1, G, part_stride(NP + 8)]; fused tail required."""
    _lib.check(_lib.load().ddrl_ppo_train_step_tc_coupled(
        _p(tc_img, torch.uint8, "tc_img"), _p(theta, torch.float32, "theta"), _p(node_id, torch.int32, "node_id"),
        *_step_args(obs, actions, old_logits, old_logp, vf_preds, adv, vtarg, A, MB, mb_perm, step_ctr, kl_coeff, hyper,
                    ctas_per_policy, grad_part, stat_part),
        _p(status, torch.int32, "status"), C.byref(tail) if tail is not None else None, _stream()), "ppo_train_step_tc_coupled")


def ppo_train_step_coupled(theta, img, node_id, obs, actions, old_logits, old_logp, vf_preds, adv, vtarg, A: int, MB: int,
                           mb_perm, step_ctr, kl_coeff, hyper: PPOHyper, ctas_per_policy: int, grad_part, stat_part,
                           tail: SgdTail):
    """Leg-coupled FP32 step (ddrl_ppo_train_step_coupled): as ppo_train_step_tc_coupled with the packed FP32 image `img`
    of the first NP entries of theta; the device flag goes to tail.status."""
    _lib.check(_lib.load().ddrl_ppo_train_step_coupled(
        _p(theta, torch.float32, "theta"), _p(img, torch.float32, "img"), _p(node_id, torch.int32, "node_id"),
        *_step_args(obs, actions, old_logits, old_logp, vf_preds, adv, vtarg, A, MB, mb_perm, step_ctr, kl_coeff, hyper,
                    ctas_per_policy, grad_part, stat_part),
        C.byref(tail) if tail is not None else None, _stream()), "ppo_train_step_coupled")


def obs_gather(obs_full: torch.Tensor, table: torch.Tensor, P: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """obs_full [S, Dfull] f32/f64, table [Ag, D] i32 -> [P, S*(Ag/P), D] f32 (agent a -> policy a // (Ag/P))."""
    S, Dfull = obs_full.shape
    Ag, D = table.shape
    if out is None:
        out = torch.empty(P, S * (Ag // P), D, dtype=torch.float32, device=obs_full.device)
    if obs_full.dtype not in (torch.float32, torch.float64):
        raise DDRLError("obs_gather: obs_full must be float32 or float64")
    _lib.check(_lib.load().ddrl_obs_gather(_p(obs_full, None, "obs_full"), int(obs_full.dtype == torch.float64), S, Dfull,
                                           _p(table, torch.int32, "table"), Ag, D, P, _p(out, torch.float32, "out"), _stream()),
               "obs_gather")
    return out


def graph_obs_build(obs_full: torch.Tensor, table: torch.Tensor, leg_zw: torch.Tensor, mean: Optional[torch.Tensor] = None,
                    std: Optional[torch.Tensor] = None, clip: float = 10.0, replicate: bool = False):
    """Node features of the shared-graph env: obs_full [S, Dfull] f32/f64 RAW, table [Ag, Dn] i32, leg_zw [Ag, 2] f64
    ({sin, cos} of half the leg angle), mean / std [Dfull] f64 frozen filter statistics (None = no normalisation)
    -> state [S, Ag, Dn+4] f32, or with ``replicate`` (state [S*Ag, Ag, Dn+4], node_idx [S*Ag] i32)."""
    S, Dfull = obs_full.shape
    Ag, Dn = table.shape
    if obs_full.dtype not in (torch.float32, torch.float64):
        raise DDRLError("graph_obs_build: obs_full must be float32 or float64")
    dev = obs_full.device
    state = torch.empty((S * Ag, Ag, Dn + 4) if replicate else (S, Ag, Dn + 4), dtype=torch.float32, device=dev)
    node_idx = torch.empty(S * Ag, dtype=torch.int32, device=dev) if replicate else None
    _lib.check(_lib.load().ddrl_graph_obs_build(_p(obs_full, None, "obs_full"), int(obs_full.dtype == torch.float64), S, Dfull,
                                                _p(table, torch.int32, "table"), Ag, Dn, _p(mean, torch.float64, "mean"),
                                                _p(std, torch.float64, "std"), float(clip), _p(leg_zw, torch.float64, "leg_zw"),
                                                int(replicate), _p(state, torch.float32, "state"),
                                                _p(node_idx, torch.int32, "node_idx"), _stream()), "graph_obs_build")
    return (state, node_idx) if replicate else state


def sgd_ll_words(P: int, ctas_per_policy: int, D: int, A: int) -> int:
    """64-bit words of the LL workspace (``ddrl_sgd_tail.ll_ws``) of the ping-pong tcgen05 step."""
    n = int(_lib.load().ddrl_sgd_ll_words(P, ctas_per_policy, D, A))
    if n <= 0:
        raise DDRLError("ddrl_sgd_ll_words failed")
    return n


def make_sgd_tail(theta, m, v, beta_pow, grad, barrier_ws, sq_ws, lr, beta1, beta2, eps, grad_clip, gnorm_out=None, img=None,
                  tc_img=None, step_stats=None, step_ctr=None, status=None, ll_ws=None, grad_acc=None) -> SgdTail:
    """Fused grad-reduce + [peer all-reduce] + clip + Adam tail of the SGD step (see ddrl_sgd_tail in ddrl_b200.h).
    The caller keeps the tensors alive; barrier_ws must be zero-initialised int32 [4*P + 4].  For world > 1 let
    ``peer.PeerExchange.fill`` add the rank / peer-buffer fields."""
    f32 = torch.float32
    t = SgdTail()
    t.theta, t.m, t.v = _p(theta, f32, "theta"), _p(m, f32, "m"), _p(v, f32, "v")
    t.beta_pow, t.grad, t.gnorm_out = _p(beta_pow, f32, "beta_pow"), _p(grad, f32, "grad"), _p(gnorm_out, f32, "gnorm_out")
    t.fcnet_img, t.fcnet_tc_img = _p(img, f32, "img"), _p(tc_img, torch.uint8, "tc_img")
    t.step_stats, t.step_ctr = _p(step_stats, torch.float64, "step_stats"), _p(step_ctr, torch.int32, "step_ctr")
    t.barrier_ws, t.sq_ws = _p(barrier_ws, torch.int32, "barrier_ws"), _p(sq_ws, f32, "sq_ws")
    t.lr, t.beta1, t.beta2, t.eps, t.grad_clip = float(lr), float(beta1), float(beta2), float(eps), float(grad_clip)
    t.status = _p(status, torch.int32, "status")
    t.world, t.rank, t.nsteps = 1, 0, 1
    t.ll_ws = _p(ll_ws, torch.int64, "ll_ws")
    t.grad_acc = _p(grad_acc, f32, "grad_acc")
    return t


REWARD_MODES = {"per_leg": 0, "per_leg_norm": 1, "global": 2, "global_costs": 3}


def reward_split(fw_reward, actions, cfrc_ext, contact_table, ctrl_cost_weight: float, contact_cost_weight: float,
                 mode: str = "per_leg"):
    """Per-agent rewards of the multi-agent adaptor, batched: fw_reward [S] f32, actions [S,Ag,A] f32, cfrc_ext [S,NB,6] f64,
    contact_table [Ag,NB] f64 -> [S,Ag] f32 (see ddrl_reward_split)."""
    S, Ag, A = actions.shape
    NB = cfrc_ext.shape[1]
    out = torch.empty(S, Ag, dtype=torch.float32, device=actions.device)
    _lib.check(_lib.load().ddrl_reward_split(_p(fw_reward, torch.float32, "fw_reward"), _p(actions, torch.float32, "actions"),
                                             _p(cfrc_ext, torch.float64, "cfrc_ext"), _p(contact_table, torch.float64, "contact_table"),
                                             S, Ag, A, NB, float(ctrl_cost_weight), float(contact_cost_weight), REWARD_MODES[mode],
                                             _p(out, torch.float32, "rewards"), _stream()), "reward_split")
    return out


def concat_actions(actions, action_table, A_full: int = 8, clip=(-1.0, 1.0)):
    """actions [S,Ag,A] f32 + action_table [Ag,A] i32 -> env actions [S,A_full] f32, clipped like RLlib's clip_actions."""
    S, Ag, A = actions.shape
    out = torch.zeros(S, A_full, dtype=torch.float32, device=actions.device)
    _lib.check(_lib.load().ddrl_concat_actions(_p(actions, torch.float32, "actions"), _p(action_table, torch.int32, "action_table"),
                                               S, Ag, A, A_full, float(clip[0]), float(clip[1]), _p(out, torch.float32, "out"),
                                               _stream()), "concat_actions")
    return out

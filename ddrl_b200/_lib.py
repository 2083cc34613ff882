"""ctypes binding of libddrl_b200.so — the same stub INTEGRATION.md gives a reference maintainer.

There is no CPU fallback: if the shared library is missing or a launch fails, every op raises."""
from __future__ import annotations

import ctypes as C
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libddrl_b200.so")

c_f32p = C.c_void_p
c_i32p = C.c_void_p
c_i64p = C.c_void_p
c_f64p = C.c_void_p
c_u8p = C.c_void_p
c_stream = C.c_void_p


class PPOHyper(C.Structure):
    _fields_ = [("clip_param", C.c_float), ("vf_clip_param", C.c_float), ("vf_loss_coeff", C.c_float),
                ("entropy_coeff", C.c_float), ("inv_global_mb", C.c_float)]


MAX_RANKS = 8


class SgdTail(C.Structure):
    _fields_ = [("theta", C.c_void_p), ("m", C.c_void_p), ("v", C.c_void_p), ("beta_pow", C.c_void_p), ("grad", C.c_void_p),
                ("gnorm_out", C.c_void_p), ("fcnet_img", C.c_void_p), ("fcnet_tc_img", C.c_void_p),
                ("step_stats", C.c_void_p), ("step_ctr", C.c_void_p), ("barrier_ws", C.c_void_p), ("sq_ws", C.c_void_p),
                ("lr", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float), ("eps", C.c_float), ("grad_clip", C.c_float),
                ("status", C.c_void_p), ("world", C.c_int32), ("rank", C.c_int32), ("seq", C.c_void_p),
                ("peer_x", C.c_void_p * MAX_RANKS), ("nsteps", C.c_int32), ("ll_ws", C.c_void_p), ("grad_acc", C.c_void_p)]


# name -> (restype, argtypes); mirrors include/ddrl_b200.h one to one (tests check every symbol).
PROTOTYPES = {
    "ddrl_last_error": (C.c_char_p, []),
    "ddrl_abi_version": (C.c_int, []),
    "ddrl_launch_count": (C.c_int64, []),
    "ddrl_fcnet_num_params": (C.c_int, [C.c_int, C.c_int]),
    "ddrl_fcnet_image_floats": (C.c_int, [C.c_int, C.c_int]),
    "ddrl_fcnet_pack": (C.c_int, [c_f32p, C.c_int, C.c_int, C.c_int, c_f32p, c_stream]),
    "ddrl_filter_ws_bytes": (C.c_int64, [C.c_int, C.c_int64, C.c_int]),
    "ddrl_filter_update": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_int, c_i64p, c_f64p, c_f64p,
                                     c_f64p, C.c_void_p, c_stream]),
    "ddrl_filter_num_partials": (C.c_int, [C.c_int64]),
    "ddrl_filter_partial": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_int, C.c_void_p, c_stream]),
    "ddrl_filter_merge": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int64, c_i64p, c_f64p, c_f64p, c_f64p,
                                    c_stream]),
    "ddrl_fcnet_forward": (C.c_int, [c_f32p, c_f32p, c_f32p, c_f64p, C.c_float, C.c_int, C.c_int64, C.c_int, C.c_int,
                                     c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_stream]),
    "ddrl_obs_gather": (C.c_int, [C.c_void_p, C.c_int, C.c_int64, C.c_int, c_i32p, C.c_int, C.c_int, C.c_int, c_f32p, c_stream]),
    "ddrl_graph_obs_build": (C.c_int, [C.c_void_p, C.c_int, C.c_int64, C.c_int, c_i32p, C.c_int, C.c_int, c_f64p, c_f64p, C.c_double,
                                       c_f64p, C.c_int, c_f32p, c_i32p, c_stream]),
    "ddrl_reward_split": (C.c_int, [c_f32p, c_f32p, c_f64p, c_f64p, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double,
                                    C.c_int, c_f32p, c_stream]),
    "ddrl_concat_actions": (C.c_int, [c_f32p, c_i32p, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, c_f32p, c_stream]),
    "ddrl_gae_ws_bytes": (C.c_int64, [C.c_int, C.c_int64]),
    "ddrl_gae": (C.c_int, [c_f32p, c_f32p, c_u8p, c_f32p, C.c_int, C.c_int, C.c_int64, C.c_int, C.c_double,
                           C.c_double, c_f32p, c_f32p, c_f64p, C.c_void_p, c_stream]),
    "ddrl_adv_standardize": (C.c_int, [c_f32p, c_f64p, C.c_int, C.c_int64, c_stream]),
    "ddrl_gather_rows": (C.c_int, [c_f32p, c_i32p, C.c_int, C.c_int64, C.c_int, c_f32p, c_stream]),
    "ddrl_ppo_train_step": (C.c_int, [c_f32p] * 11 + [C.c_int, C.c_int64, C.c_int, C.c_int, C.c_int, c_i32p,
                                                     C.c_int64, c_i32p, c_f32p, C.POINTER(PPOHyper), C.c_int,
                                                     c_f32p, c_f64p, C.POINTER(SgdTail), c_stream]),
    "ddrl_ppo_loss_grad": (C.c_int, [c_f32p] * 8 + [C.c_int, C.c_int64, C.c_int, c_f32p, C.POINTER(PPOHyper), C.c_int,
                                                    c_f32p, c_f32p, c_f64p, c_stream]),
    "ddrl_grad_reduce": (C.c_int, [c_f32p, c_f64p, C.c_int, C.c_int, C.c_int, c_f32p, c_f64p, c_i32p, c_stream]),
    "ddrl_clip_adam": (C.c_int, [c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, C.c_int, C.c_int, C.c_float, C.c_float,
                                 C.c_float, C.c_float, C.c_float, c_f32p, c_i32p, c_i32p, c_f32p, C.c_void_p, C.c_int,
                                 C.c_int, c_stream]),
    "ddrl_graphnet_num_params": (C.c_int, [C.c_int]),
    "ddrl_graphnet_set_variant": (C.c_int, [C.c_int]),
    "ddrl_graphnet_train_ws_bytes": (C.c_int64, [C.c_int64]),
    "ddrl_graphnet_train_stat_parts": (C.c_int, [C.c_int64]),
    "ddrl_graphnet_train_step_tc": (C.c_int, [c_f32p, c_i32p] + [c_f32p] * 8 + [C.c_int64, C.c_int, C.c_int, c_i32p, c_i32p, c_f32p,
                                                C.POINTER(PPOHyper), C.c_int, c_f32p, c_f64p, c_i32p, C.POINTER(SgdTail), c_stream]),
    "ddrl_graphnet_train_step": (C.c_int, [c_f32p, c_i32p, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p,
                                           C.c_int64, C.c_int, c_f32p, C.POINTER(PPOHyper), C.c_int, C.c_void_p, c_f32p, c_f64p,
                                           c_stream]),
    "ddrl_graphnet_forward": (C.c_int, [c_f32p, c_i32p, c_f32p, c_f32p, C.c_int64, C.c_int, c_f32p, c_f32p,
                                        c_stream]),
    "ddrl_graphnet_act": (C.c_int, [c_f32p, c_i32p, c_f32p, c_f32p, c_f32p, C.c_int64, C.c_int, c_f32p, c_f32p, c_f32p,
                                    c_f32p, c_stream]),
    "ddrl_graphnet_backward": (C.c_int, [c_f32p, c_i32p, c_f32p, c_f32p, c_f32p, c_f32p, C.c_int64, C.c_int,
                                         C.c_int, c_f32p, c_stream]),
    "ddrl_gcn_forward": (C.c_int, [c_f32p, c_f32p, c_f32p, c_f32p, C.c_int64, C.c_int, C.c_int, C.c_int, c_f32p,
                                   c_stream]),
    "ddrl_dg_sample": (C.c_int, [c_f32p, c_f32p, C.c_int64, C.c_int, c_f32p, c_f32p, c_stream]),
    "ddrl_leg_coupling": (C.c_int, [c_f32p, c_i32p, c_f32p, C.c_int64, C.c_int, c_stream]),
    "ddrl_param_expand": (C.c_int, [c_f32p, c_i32p, C.c_int, C.c_int, C.c_int, c_f32p, c_stream]),
    "ddrl_grad_tie": (C.c_int, [c_f32p, c_i32p, C.c_int, C.c_int, C.c_int, c_f32p, c_stream]),
    "ddrl_leg_coupling_backward": (C.c_int, [c_f32p, c_f32p, c_i32p, c_f32p, C.c_int64, C.c_int, c_f32p, c_stream]),
    "ddrl_fcnet_tc_image_bytes": (C.c_int, [C.c_int, C.c_int]),
    "ddrl_fcnet_train_supported": (C.c_int, [C.c_int, C.c_int, C.c_int]),
    "ddrl_fcnet_forward_tc": (C.c_int, [C.c_void_p, c_f32p, c_f64p, C.c_float, C.c_int, C.c_int64, C.c_int, C.c_int,
                                         c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_i32p, c_stream]),
    "ddrl_fcnet_forward_coupled": (C.c_int, [c_f32p, c_f32p, c_i32p, c_f32p, c_f32p, c_f64p, C.c_float, C.c_int, C.c_int64,
                                             C.c_int, C.c_int, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_i32p, c_stream]),
    "ddrl_fcnet_forward_tc_coupled": (C.c_int, [C.c_void_p, c_i32p, c_f32p, c_f32p, c_f64p, C.c_float, C.c_int, C.c_int64,
                                                C.c_int, C.c_int, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_f32p, c_i32p,
                                                c_stream]),
    "ddrl_tc_set_variant": (C.c_int, [C.c_int]),
    "ddrl_mpnn2_forward": (C.c_int, [c_f32p] * 5 + [C.c_int64, C.c_int, C.c_int, C.c_int, c_f32p, c_stream]),
    "ddrl_gat1_forward": (C.c_int, [c_f32p] * 5 + [C.c_int64, C.c_int, C.c_int, C.c_int, c_f32p, c_stream]),
    "ddrl_mpnn2_backward": (C.c_int, [c_f32p] * 6 + [C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int, c_f32p, c_f32p, c_stream]),
    "ddrl_gat1_backward": (C.c_int, [c_f32p] * 6 + [C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int, c_f32p, c_f32p, c_stream]),
    "ddrl_symm_norm": (C.c_int, [c_f32p, C.c_int64, C.c_int, c_f32p, c_stream]),
    "ddrl_segment_softmax": (C.c_int, [c_f32p, c_i32p, C.c_int64, C.c_int, C.c_int64, c_f32p, c_i32p, c_f32p, c_stream]),
    "ddrl_tc_pingpong_eligible": (C.c_int, [C.c_int, C.c_int]),
    "ddrl_tc_set_cluster": (C.c_int, [C.c_int]),
    "ddrl_tc_last_cluster": (C.c_int, []),
    "ddrl_tc_set_debug_clock": (C.c_int, [C.c_void_p]),
    "ddrl_umma_bench": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, c_i32p, c_stream]),
    "ddrl_sgd_exchange_words": (C.c_int64, [C.c_int, C.c_int]),
    "ddrl_sgd_ll_words": (C.c_int64, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "ddrl_peer_alloc": (C.c_int, [C.c_int64, C.POINTER(C.c_void_p), C.c_void_p]),
    "ddrl_peer_open": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "ddrl_peer_close": (C.c_int, [C.c_void_p]),
    "ddrl_peer_free": (C.c_int, [C.c_void_p]),
    "ddrl_fcnet_tc_pack": (C.c_int, [c_f32p, C.c_int, C.c_int, C.c_int, C.c_void_p, c_stream]),
    "ddrl_ppo_train_step_tc": (C.c_int, [C.c_void_p] + [c_f32p] * 7 + [C.c_int, C.c_int64, C.c_int, C.c_int, C.c_int, c_i32p,
                                                                     C.c_int64, c_i32p, c_f32p, C.POINTER(PPOHyper), C.c_int,
                                                                     c_f32p, c_f64p, c_i32p, C.POINTER(SgdTail), c_stream]),
    "ddrl_ppo_train_step_coupled": (C.c_int, [c_f32p, c_f32p, c_i32p] + [c_f32p] * 7 + [C.c_int, C.c_int64, C.c_int, C.c_int, C.c_int,
                                                                             c_i32p, C.c_int64, c_i32p, c_f32p, C.POINTER(PPOHyper),
                                                                             C.c_int, c_f32p, c_f64p, C.POINTER(SgdTail), c_stream]),
    "ddrl_ppo_train_step_tc_coupled": (C.c_int, [C.c_void_p, c_f32p, c_i32p] + [c_f32p] * 7 +
                                       [C.c_int, C.c_int64, C.c_int, C.c_int, C.c_int, c_i32p, C.c_int64, c_i32p, c_f32p,
                                        C.POINTER(PPOHyper), C.c_int, c_f32p, c_f64p, c_i32p, C.POINTER(SgdTail), c_stream]),
    "ddrl_umma_selftest": (C.c_int, [c_f32p, C.c_int, C.c_int, c_f32p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                     C.c_int, C.c_int, c_f32p, c_i32p, c_stream]),
}

_lib = None


class DDRLError(RuntimeError):
    pass


def load():
    """Load the C-ABI library (once).  Raises if it has not been built — no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise DDRLError(
                f"{LIB_PATH} is missing: build it with `python -m ddrl_b200.build` (nvcc, sm_100a). "
                "ddrl_b200 has no CPU or PyTorch fallback.")
        lib = C.CDLL(os.environ.get("DDRL_B200_LIB", LIB_PATH))   # override: A/B timing of alternative builds
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().ddrl_last_error().decode("utf-8", "replace")
        raise DDRLError(f"{what or 'ddrl'} failed (code {rc}): {msg}")

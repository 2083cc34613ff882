"""Shared helpers for the tests (golden fixture loading, synthetic rollouts).  Test infrastructure only."""
import json
import os

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")

# (arch file stem) -> (policy order used by the env's policy_names, D, A)
ARCHS = {
    "Centralized": (["central_policy"], 43, 8),
    "FullyDecentral": (["policy_FL", "policy_HL", "policy_HR", "policy_FR"], 19, 2),
    "Local": (["policy_FL", "policy_HL", "policy_HR", "policy_FR"], 35, 2),
    "SingleDiagonal": (["policy_FL", "policy_HL", "policy_HR", "policy_FR"], 27, 2),
    "SingleNeighbor": (["policy_FL", "policy_HL", "policy_HR", "policy_FR"], 27, 2),
    "SingleToFront": (["policy_FL", "policy_HL", "policy_HR", "policy_FR"], 27, 2),
    "TwoDiags": (["policy_FLHR", "policy_HLFR"], 27, 4),
    "TwoSides": (["policy_LEFT", "policy_RIGHT"], 27, 4),
    "Centralized_TVel": (["central_policy"], 44, 8),
    "FullyDecentral_TVel": (["policy_FL", "policy_HL", "policy_HR", "policy_FR"], 20, 2),
    "Local_TVel": (["policy_FL", "policy_HL", "policy_HR", "policy_FR"], 36, 2),
    "TwoSides_TVel": (["policy_LEFT", "policy_RIGHT"], 28, 4),
}


def load_ckpt(arch):
    return np.load(os.path.join(GOLDEN, f"ckpt_{arch}.npz"))


def ckpt_theta(arch):
    """-> theta [P, NP] float32 in the env's policy order, filters list of (n, M, S)."""
    pids, D, A = ARCHS[arch]
    z = load_ckpt(arch)
    theta = np.stack([z[f"{pid}/theta"] for pid in pids])
    filt = [(int(z[f"{pid}/filter_n"]), z[f"{pid}/filter_M"], z[f"{pid}/filter_S"]) for pid in pids]
    return theta, filt, D, A


def learner_stats():
    return json.load(open(os.path.join(GOLDEN, "learner_stats.json")))


def synth_obs(filt, R, seed):
    """raw observations ~ N(mean, std^2) of a checkpoint filter (SURVEY.md §8-d) -> [P, R, D] float32."""
    rng = np.random.default_rng(seed)
    out = []
    for n, M, S in filt:
        std = np.sqrt(S / (n - 1))
        out.append((M + std * rng.standard_normal((R, M.shape[0]))).astype(np.float32))
    return np.stack(out)


def rel_err(a, b, floor=1e-6):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b) / (np.abs(b) + floor))) if a.size else 0.0


def scaled_err(a, b):
    """max |a-b| / max|b| : error relative to the tensor's scale (robust for entries near zero)."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / (np.max(np.abs(b)) + 1e-30)) if a.size else 0.0


def t64(x):
    return torch.from_numpy(np.asarray(x, dtype=np.float64))


def assert_grad_per_variable(grad, ref, twin, shapes, gtol, where=(), allow=None):
    """Per-variable gradient check, so that a small tensor (biases, heads) cannot hide behind a large one.  grad: the kernel's
    flat gradient, ref: float64 autograd, twin: float32 autograd of the same loss; shapes: the variables' shapes in flat order.
    A bias gradient is a cancelling sum over rows (e.g. value_out/bias = sum_r dL/dv_r ~ 3e-4 from terms ~ 2e-2): perturbing
    v by 3 ulp moves it by 1e-3 relative, so its own magnitude is not a usable scale for FP32 round-off.  Each variable is
    held to 2 * gtol of max(own scale, 1 % of the whole gradient's scale; 5 % for 1-D variables, which are pure cancelling
    sums), or 4x the float32 twin's error.  allow: {flat offset of a variable: absolute error it may have} for a variable
    whose error the caller bounds from its own derivation."""
    grad, ref, twin = (np.asarray(a, dtype=np.float64) for a in (grad, ref, twin))
    gscale = np.abs(ref).max()
    o = 0
    for shp in shapes:
        n = int(np.prod(shp))
        err = np.abs(grad[o:o + n] - ref[o:o + n]).max()
        e_twin = np.abs(twin[o:o + n] - ref[o:o + n]).max()
        scale = max(np.abs(ref[o:o + n]).max(), (0.05 if len(shp) == 1 else 0.01) * gscale)
        lim = max(2.0 * gtol * scale, 4.0 * e_twin, (allow or {}).get(o, 0.0))
        assert err < lim, (*where, "variable at", o, tuple(shp), err, scale, e_twin)
        o += n
    assert o == ref.size, (o, ref.size)

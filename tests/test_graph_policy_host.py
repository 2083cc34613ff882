"""CPU: the host half of the shared GraphNet policy's RLlib surface — validation of the Tuple observation
(node_idx, state, adj) and, in a subprocess, `GraphNetPolicyGroup`'s orchestration with every kernel replaced by the oracle
(tests/host_dryrun_graph_policy.py)."""
import os
import subprocess
import sys

import numpy as np
import pytest

from ddrl_b200 import rllib_policy as RP


def _obs(B, seed=0):
    rng = np.random.default_rng(seed)
    return (rng.integers(0, 4, size=B), rng.standard_normal((B, 4, 23)),
            (rng.random((B, 4, 4)) < 0.5).astype(np.int64))


def test_check_graph_obs_accepts_the_env_spaces():
    idx, state, adj = _obs(9)
    node, st, a = RP.check_graph_obs(idx[:, None], state, adj, "p")            # [B, 1] node ids, float64 state, int adj
    assert node.dtype == np.int32 and np.array_equal(node, idx)
    assert st.dtype == np.float32 and st.flags.c_contiguous and np.array_equal(st, state.astype(np.float32))
    assert a.dtype == np.float32 and np.array_equal(a, adj)
    node, st, a = RP.check_graph_obs(idx.astype(np.float32), state.astype(np.float32), adj.astype(bool), "p")
    assert np.array_equal(node, idx) and np.array_equal(a, adj)
    assert RP.check_graph_obs(idx[:0], state[:0], adj[:0], "p")[1].shape == (0, 4, 23)


@pytest.mark.parametrize("what", ["node 4", "node -1", "node 1.5", "node rows", "adj 2", "adj 0.5", "adj NaN", "adj shape",
                                  "state NaN", "state inf", "state shape", "state width 19", "state int"])
def test_check_graph_obs_rejects(what):
    idx, state, adj = _obs(8, 1)
    idx, state, adj = idx.copy(), state.copy(), adj.astype(np.float64)
    if what == "node 4":
        idx[3] = 4
    elif what == "node -1":
        idx[0] = -1
    elif what == "node 1.5":
        idx = idx + 0.5
    elif what == "node rows":
        idx = idx[:-1]
    elif what == "adj 2":
        adj[2, 1, 0] = 2
    elif what == "adj 0.5":
        adj[0, 0, 0] = 0.5
    elif what == "adj NaN":
        adj[1, 2, 3] = np.nan
    elif what == "adj shape":
        adj = adj[:, :3]
    elif what == "state NaN":
        state[4, 2, 7] = np.nan
    elif what == "state inf":
        state[4, 2, 7] = 1e39                  # finite in float64, inf in float32
    elif what == "state shape":
        state = state.reshape(8, 92)
    elif what == "state width 19":
        state = state[..., :19]
    elif what == "state int":
        state = state.astype(np.int64)
    with pytest.raises(RP.BatchError):
        RP.check_graph_obs(idx, state, adj, "p")


def test_graph_policy_orchestration_with_oracle_mocked_kernels():
    """tests/host_dryrun_graph_policy.py: the GPU test of `GraphNetPolicyGroup`'s RLlib calls executed on CPU with the
    kernels and the SGD phase replaced by the oracle — host orchestration only (own process: it monkeypatches torch)."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "tests", "host_dryrun_graph_policy.py")], capture_output=True,
                         text=True, timeout=900, cwd=root)
    assert out.returncode == 0, out.stdout[-1500:] + out.stderr[-3000:]
    assert out.stdout.split() == ["tc", "ok", "three-kernel", "ok"]

"""GPU: ddrl_filter_stream (csrc/filter_stream.cu) against RLlib's row-by-row sampler filtering
(tests/filter_stream_oracle.py), and the learner / RLlib-facing surface in filter_mode="stream".

Bounds of the kernel:
  - every float32 row within the larger of 2 float32 ulps and 1e-10 * (|x| + |M|) / (std + 1e-8): a chunk starts from a
    merged prefix state (1e-12 relative of the sequential one), and that error is carried through the subtraction and
    the division.  The first chunk of every stream is walked from the running state itself: bit for bit;
  - merged count bit-exact, mean / M2 within 1e-12 relative of the sequential order (DESIGN.md §2);
  - two launches bit-identical."""
import os
import socket
import time

import numpy as np
import pytest
import torch

from tests.filter_stream_oracle import StreamFilter, filter_stream, running_stat, state_error_bound, stream_rows
from tests.util import ckpt_theta, scaled_err, synth_obs

pytestmark = pytest.mark.gpu

CHUNK = 64      # FS_CHUNK of the kernel
TOL = 1e-5


def _oracle():
    import oracle.ddrl_oracle as O
    return O


def _dev(a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a))
    return (t.to(dtype) if dtype is not None else t).cuda()


def _start(kind, P, D, rng):
    """(n [P], M [P, D], S [P, D]): empty, small, or warm — the filters of a published checkpoint (n ~ 2e7)."""
    if kind == "empty":
        return np.zeros(P, np.int64), np.zeros((P, D)), np.zeros((P, D))
    if kind == "small":
        return (np.array([1 + p for p in range(P)], np.int64), rng.standard_normal((P, D)),
                rng.uniform(0.2, 3.0, (P, D)))
    _, filt, _, _ = ckpt_theta("Centralized_TVel" if D > 19 else "FullyDecentral")
    n = np.array([filt[p % len(filt)][0] for p in range(P)], np.int64)
    rep = lambda v: np.resize(v, D)
    return n, np.stack([rep(filt[p % len(filt)][1]) for p in range(P)]), np.stack([rep(filt[p % len(filt)][2]) for p in range(P)])


def _rows(P, R, D, start, rng):
    n, M, S = start
    std = np.where(n[:, None] > 1, np.sqrt(S / np.maximum(n[:, None] - 1, 1)), 1.0) + 0.3
    return (M[:, None, :] + 1.5 * std[:, None, :] * rng.standard_normal((P, R, D)))


def _check_kernel(x, T, C, W, start, clip, f64=False):
    """Runs the kernel twice on x [P, R, D] and checks it against the oracle per policy."""
    from ddrl_b200 import kernels as K
    P, R, D = x.shape
    xs = x.astype(np.float64 if f64 else np.float32)
    n, M, S = (_dev(start[0]), _dev(start[1]), _dev(start[2]))
    xd = _dev(xs)
    out, parts = K.filter_stream(xd, n, M, S, T, W, clip)
    out2, parts2 = K.filter_stream(xd, n, M, S, T, W, clip)
    norm = torch.empty(P, 2, D, dtype=torch.float64, device="cuda")
    K.filter_merge(parts, R, n, M, S, norm)
    torch.cuda.synchronize()
    assert torch.equal(out, out2) and torch.equal(parts, parts2)
    out, parts = out.cpu().numpy(), parts.cpu().numpy()
    for p in range(P):
        st = (int(start[0][p]), start[1][p], start[2][p])
        y, drv, bufs, mean, std = filter_stream(xs[p], T, C, W, st, clip or None, row_state=True)
        y32 = y.astype(np.float32)
        ulp = np.spacing(np.abs(y32)).astype(np.float64)
        bound = np.maximum(2 * ulp, state_error_bound(xs[p], mean, std))
        err = np.abs(out[p].astype(np.float64) - y32)
        assert np.all(err <= bound), (p, float((err / bound).max()))
        for rows in stream_rows(T, C, W):
            first = rows[:CHUNK]
            np.testing.assert_array_equal(out[p][first], y32[first])
        for w, b in enumerate(bufs):
            assert parts[p, w, 0, 0] == b.n
            np.testing.assert_allclose(parts[p, w, :, 1], b.mean, rtol=1e-12, atol=1e-12 * np.abs(b.mean).max())
            np.testing.assert_allclose(parts[p, w, :, 2], b._S, rtol=1e-12)
        assert int(n[p]) == drv.n
        np.testing.assert_allclose(M[p].cpu().numpy(), drv.mean, rtol=1e-12, atol=1e-12 * np.abs(drv.mean).max())
        np.testing.assert_allclose(S[p].cpu().numpy(), drv._S, rtol=1e-12)


@pytest.mark.parametrize("start", ["empty", "small", "warm"])
@pytest.mark.parametrize("clip", [0.0, 10.0])
@pytest.mark.parametrize("f64", [False, True])
@pytest.mark.parametrize("W", [1, 2, 4])
@pytest.mark.parametrize("D", [19, 43, 64])
@pytest.mark.parametrize("P", [1, 4])
def test_kernel_matches_row_by_row_filter(P, D, W, f64, clip, start):
    """T = 9, C = 40: 360 rows per policy, not a multiple of the 64-row chunk; W = 4 streams of 90 rows (two chunks)."""
    rng = np.random.default_rng(P * 1000 + D * 10 + W)
    T, C = 9, 40
    st = _start(start, P, D, rng)
    _check_kernel(_rows(P, T * C, D, st, rng), T, C, W, st, clip, f64)


@pytest.mark.parametrize("T,C,W,P,D", [(100, 4, 4, 2, 19),        # four one-column streams
                                       (40, 200, 1, 1, 19),        # 125 chunks: several chunks per scan group
                                       (3, 7, 7, 1, 5),            # streams shorter than one chunk
                                       (32, 4096, 1, 1, 19),       # the bench shape (one policy of it)
                                       (32, 4096, 2, 1, 19)])
def test_kernel_on_ragged_one_column_and_bench_shapes(T, C, W, P, D):
    rng = np.random.default_rng(T + C + W)
    for start in ("empty", "warm"):
        st = _start(start, P, D, rng)
        _check_kernel(_rows(P, T * C, D, st, rng), T, C, W, st, 0.0)


def test_error_codes():
    from ddrl_b200 import _lib
    lib = _lib.load()
    x = torch.zeros(1, 12, 4, device="cuda")
    n = torch.zeros(1, dtype=torch.int64, device="cuda")
    M = torch.zeros(1, 4, dtype=torch.float64, device="cuda")
    out = torch.empty(1, 12, 4, device="cuda")
    parts = torch.empty(1, 4, 4, 3, dtype=torch.float64, device="cuda")
    ws = torch.empty(1 << 16, dtype=torch.uint8, device="cuda")
    s = torch.cuda.current_stream().cuda_stream

    def call(P=1, T=2, C=6, W=2, D=4, x_=x, ws_=ws):
        return lib.ddrl_filter_stream(x_.data_ptr() if x_ is not None else None, 0, P, T, C, W, D, n.data_ptr(), M.data_ptr(),
                                      M.data_ptr(), 0.0, out.data_ptr(), parts.data_ptr(),
                                      ws_.data_ptr() if ws_ is not None else None, s)
    assert call() == 0
    assert call(W=4) == -1                      # C % W != 0
    for bad in (dict(P=0), dict(T=0), dict(C=0), dict(W=0), dict(D=0), dict(x_=None), dict(ws_=None)):
        assert call(**bad) == -1, bad
    assert call(D=65) == -2
    assert lib.ddrl_filter_stream_ws_bytes(1, 2, 6, 4, 4) == -1
    assert lib.ddrl_filter_stream_ws_bytes(1, 2, 6, 2, 4) == 1 * 2 * 1 * 4 * 3 * 8
    torch.cuda.synchronize()


# ---- the learner ------------------------------------------------------------------------------------------------------------

def _problem(arch, T, C, seed):
    theta0, filt, D, A = ckpt_theta(arch)
    P = theta0.shape[0]
    rng = np.random.default_rng(seed)
    filt0 = [(1000, M, S * (999.0 / (n - 1))) for n, M, S in filt]
    raw = synth_obs(filt, T * C, seed).reshape(P, T, C, D)
    boot = synth_obs(filt, C, seed + 1)
    rewards = (0.3 + 0.5 * rng.standard_normal((P, T, C))).astype(np.float32)
    dones = (rng.random((T, C)) < 0.05).astype(np.uint8)
    eps = rng.standard_normal((P, T, C, A)).astype(np.float32)
    return dict(theta0=theta0, filt0=filt0, D=D, A=A, P=P, raw=raw, boot=boot, rewards=rewards, dones=dones, eps=eps, rng=rng)


def _set_filter(L, filt0):
    L.filt_n.copy_(torch.tensor([f[0] for f in filt0]))
    L.filt_M.copy_(torch.from_numpy(np.stack([f[1] for f in filt0])))
    L.filt_S.copy_(torch.from_numpy(np.stack([f[2] for f in filt0])))


@pytest.mark.parametrize("mode", ["fp32", "tc"])
@pytest.mark.parametrize("W", [1, 2])
def test_learner_iteration_matches_oracle_with_stream_filter(mode, W):
    """One learn_on_rollout iteration in filter_mode="stream" against the oracle iteration with the row-by-row worker
    filtering swapped in: filter state to 1e-12, stored obs / logits / values to 1e-5, weights no further from float64
    than 10x the float32 twin."""
    from ddrl_b200.config import PPOConfig
    from ddrl_b200.learner import FCNetLearner
    O = _oracle()
    T, C, MB = 16, 32, 128
    pr = _problem("FullyDecentral", T, C, 6)
    P, D, A, rng = pr["P"], pr["D"], pr["A"], pr["rng"]
    R = T * C
    cfgd = dict(num_sgd_iter=2, sgd_minibatch_size=MB)
    perms = np.stack([np.stack([rng.permutation(R // MB) for _ in range(2)]) for _ in range(P)]).astype(np.int32)
    shuffle = np.stack([rng.permutation(R) for _ in range(P)]).astype(np.int32)
    L = FCNetLearner(P, D, A, PPOConfig(**cfgd), "cuda", theta=torch.from_numpy(pr["theta0"]), mode=mode,
                     filter_mode="stream", filter_workers=W)
    _set_filter(L, pr["filt0"])
    stats = L.learn_on_rollout(_dev(pr["raw"]), _dev(pr["boot"]), _dev(pr["rewards"]), _dev(pr["dones"]), _dev(pr["eps"]),
                               _dev(perms), _dev(shuffle))
    torch.cuda.synchronize()
    cfg_o = O.PPOConfig(**cfgd)
    runs = {}
    for dt in (torch.float64, torch.float32):
        pols = [O.PolicyState(torch.from_numpy(pr["theta0"][p].copy()).to(dt), O.AdamState.zeros(pr["theta0"].shape[1], dt, cfg_o),
                              StreamFilter(D, pr["filt0"][p], T, C, W), cfg_o.kl_coeff) for p in range(P)]
        runs[dt] = (pols, O.fcnet_learner_iteration(pols, pr["raw"], pr["boot"], pr["rewards"], pr["dones"], pr["eps"], shuffle,
                                                    perms, 2 * A, cfg_o, dt))
    (pols, out), (twin, _) = runs[torch.float64], runs[torch.float32]
    b = L._bufs
    for p in range(P):
        assert int(L.filt_n[p]) == pols[p].filt.rs.n == 1000 + R
        np.testing.assert_allclose(L.filt_M[p].cpu().numpy(), pols[p].filt.rs.mean, rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(L.filt_S[p].cpu().numpy(), pols[p].filt.rs._S, rtol=1e-12)
        assert scaled_err(b["obs"][p].cpu().numpy(), out[p]["obs_norm"]) < 1e-6
        for k_dev, k_ref in (("logits", "logits"), ("value", "value"), ("act", "actions"), ("logp", "logp")):
            assert scaled_err(b[k_dev][p].cpu().numpy(), out[p][k_ref].numpy()) < TOL, k_dev
        assert scaled_err(b["vtarg"][p].cpu().numpy(), out[p]["value_targets"].reshape(-1)) < TOL
        upd_o = pols[p].theta.numpy() - pr["theta0"][p]
        err_dev = scaled_err(L.theta[p].cpu().numpy().astype(np.float64) - pr["theta0"][p], upd_o)
        err_twin = scaled_err(twin[p].theta.numpy().astype(np.float64) - pr["theta0"][p], upd_o)
        assert err_dev < 10.0 * err_twin + 1e-5, (err_dev, err_twin)
        for k in ("policy_loss", "vf_loss", "kl", "entropy"):
            ref = out[p]["stats"][k]
            assert abs(stats[p][k] - ref) < 1e-4 * max(1.0, abs(ref)), (k, stats[p][k], ref)


@pytest.mark.parametrize("mode", ["fp32", "tc"])
def test_coupled_learner_iteration_matches_oracle_with_stream_filter(mode):
    """The leg-coupled policy (SharedDecentralLegID), 2 workers over 8 envs x 4 legs."""
    from ddrl_b200.config import PPOConfig
    from ddrl_b200.learner import FCNetLearner
    from tests.coupling_oracle import coupled_learner_iteration
    from tests.test_gpu_coupling_learner import TABLE, _rollout
    O = _oracle()
    T, N, E, MB, W = 16, 8, 2, 128, 2
    C, R = 4 * N, 16 * 4 * N
    th0 = torch.cat([O.fcnet_init(19, 4, torch.Generator().manual_seed(7)), torch.from_numpy(TABLE.reshape(-1))])
    L = FCNetLearner(1, 19, 2, PPOConfig(num_sgd_iter=E, sgd_minibatch_size=MB), "cuda", theta=th0[None], mode=mode,
                     leg_coupling=True, atomic_reduce=False, filter_mode="stream", filter_workers=W)
    raw, boot, rew, denv, eps = _rollout(T, N, 3)
    rng = np.random.default_rng(5)
    sh = rng.permutation(R).astype(np.int32)
    perms = np.stack([rng.permutation(R // MB) for _ in range(E)]).astype(np.int32)
    L.learn_on_rollout(_dev(raw[None]), _dev(boot[None]), _dev(rew[None]), _dev(denv), _dev(eps[None]), _dev(perms[None]),
                       shuffle=_dev(sh[None]), cols_per_env=4)
    torch.cuda.synchronize()
    cfg_o = O.PPOConfig(num_sgd_iter=E, sgd_minibatch_size=MB)
    traj = {}
    for dt in (torch.float64, torch.float32):
        ps = O.PolicyState(th0.to(dt).clone(), O.AdamState.zeros(th0.numel(), dt, cfg_o),
                           StreamFilter(19, (0, np.zeros(19), np.zeros(19)), T, C, W), cfg_o.kl_coeff)
        traj[dt] = (ps, coupled_learner_iteration(ps, raw, boot, rew, np.repeat(denv, 4, axis=1), eps, sh, perms, cfg_o, dt))
    (ref, res), (twin, _) = traj[torch.float64], traj[torch.float32]
    assert int(L.filt_n[0]) == ref.filt.rs.n == R
    np.testing.assert_allclose(L.filt_M[0].cpu().numpy(), ref.filt.rs.mean, rtol=1e-12, atol=1e-12)
    b = L._bufs
    assert scaled_err(b["logits"][0].cpu().numpy(), res["logits"].numpy()) < TOL
    assert scaled_err(b["value"][0].cpu().numpy(), res["value"].numpy()) < TOL
    upd = float((ref.theta - th0.double()).abs().max())
    e_dev = float((L.theta[0].cpu().double() - ref.theta).abs().max())
    e_twin = float((twin.theta.double() - ref.theta).abs().max())
    assert e_dev <= 10 * e_twin + 1e-4 * upd, (e_dev, e_twin, upd)


def test_captured_prepare_phase_is_bit_identical_to_eager():
    """use_graph=True captures the preparation phase (stream filter, merge, forward, GAE, shuffle) and replays it: three
    iterations leave exactly the state of the eager learner (fixed-order gradient reduction)."""
    from ddrl_b200.config import PPOConfig
    from ddrl_b200.learner import FCNetLearner
    T, C = 16, 32
    pr = _problem("FullyDecentral", T, C, 9)
    P, D, A, rng = pr["P"], pr["D"], pr["A"], pr["rng"]
    R = T * C
    perms = _dev(np.stack([np.stack([rng.permutation(R // 128) for _ in range(2)]) for _ in range(P)]).astype(np.int32))
    shuffle = _dev(np.stack([rng.permutation(R) for _ in range(P)]).astype(np.int32))
    args = (_dev(pr["raw"]), _dev(pr["boot"]), _dev(pr["rewards"]), _dev(pr["dones"]), _dev(pr["eps"]), perms, shuffle)
    out = []
    for graph in (True, False):
        L = FCNetLearner(P, D, A, PPOConfig(num_sgd_iter=2, sgd_minibatch_size=128), "cuda",
                         theta=torch.from_numpy(pr["theta0"]), use_graph=graph, atomic_reduce=False, filter_mode="stream",
                         filter_workers=2)
        stats = [L.learn_on_rollout(*args) for _ in range(3)]
        torch.cuda.synchronize()
        if graph:
            assert L._prep_graphs is not None and len(L._prep_graphs) == 1, getattr(L, "graph_error", None)
        out.append((L.theta.clone(), L.filt_n.clone(), L.filt_M.clone(), L.filt_S.clone(), L._bufs["obs"].clone(), stats))
    for x, y in zip(out[0][:5], out[1][:5]):
        assert torch.equal(x, y)
    assert out[0][5] == out[1][5]


def test_batch_mode_stays_the_default_and_rejects_bad_worker_splits():
    from ddrl_b200._lib import DDRLError
    from ddrl_b200.config import PPOConfig
    from ddrl_b200.learner import FCNetLearner
    L = FCNetLearner(1, 19, 2, PPOConfig(), "cuda")
    assert L.filter_mode == "batch" and L.filter_workers == 1
    with pytest.raises(DDRLError):
        FCNetLearner(1, 19, 2, PPOConfig(), "cuda", filter_mode="rows")
    L = FCNetLearner(1, 19, 2, PPOConfig(num_sgd_iter=1, sgd_minibatch_size=8), "cuda", filter_mode="stream", filter_workers=3)
    z = lambda *s: torch.zeros(*s, device="cuda")
    with pytest.raises(DDRLError, match="filter_workers"):
        L.learn_on_rollout(z(1, 2, 8, 19), z(1, 8, 19), z(1, 2, 8), torch.zeros(2, 8, dtype=torch.uint8, device="cuda"),
                           z(1, 2, 8, 2), torch.zeros(1, 1, 2, dtype=torch.int32, device="cuda"))


@pytest.mark.parametrize("scope", ["FullyDecentral", "SharedDecentralLegID"])
def test_policy_group_compute_actions_is_an_rllib_rollout_worker(scope):
    """A sequence of PPOPolicyGroup.compute_actions(update_filter=True) calls in stream mode equals RLlib's per-row sampler
    loop: the filter state to 1e-12, logits / values / actions to 1e-5 of the forward on the oracle's rows."""
    from ddrl_b200.rllib_policy import PPOPolicyGroup
    O = _oracle()
    grp = PPOPolicyGroup("QuantrupedMultiEnv_" + scope, {}, seed=3, filter_mode="stream")
    L, D, A = grp.learner, grp.D, grp.A
    L.theta.copy_(0.2 * torch.randn(L.theta.shape, generator=torch.Generator().manual_seed(1)).cuda())
    P = len(grp.policy_names)
    filt = [O.MeanStdFilter((D,), clip=None) for _ in range(P)]
    rng = np.random.default_rng(4)
    th = L.theta.cpu().double()
    for B in (1, 7, 64, 200):
        raw = (rng.standard_normal((P, B, D)) * 2.0 + 0.7).astype(np.float32)
        if grp.coupled:
            node = (np.arange(B) % 4).astype(np.int32)
            res = grp.compute_actions({grp.policy_names[0]: (node, raw[0])}, explore=False, update_filter=True)
        else:
            res = grp.compute_actions({pid: raw[i] for i, pid in enumerate(grp.policy_names)}, explore=False, update_filter=True)
        for i, pid in enumerate(grp.policy_names):
            y = np.stack([filt[i](raw[i, b]) for b in range(B)])          # one unvectorised call per row
            x = torch.from_numpy(y.astype(np.float32)).double()
            lg, v = O.fcnet_forward(th[i, :L.NPf], x, 2 * A)
            if grp.coupled:
                lg = O.leg_coupling(lg, torch.from_numpy(node.astype(np.int64)), th[i, L.NPf:].reshape(4, 2))
            act, _, info = res[pid]
            assert scaled_err(info["action_dist_inputs"], lg.numpy()) < TOL
            assert scaled_err(info["vf_preds"], v.numpy()) < TOL
            assert scaled_err(act, lg[:, :A].numpy()) < TOL
            assert int(L.filt_n[i]) == filt[i].rs.n
            np.testing.assert_allclose(L.filt_M[i].cpu().numpy(), filt[i].rs.mean, rtol=1e-12, atol=1e-12)
            np.testing.assert_allclose(L.filt_S[i].cpu().numpy(), filt[i].rs._S, rtol=1e-12, atol=1e-300)


# ---- world 2 ------------------------------------------------------------------------------------------------------------------
MT, MC, ME, MNB, MW = 16, 64, 2, 4, 2


def _multi_learner(pr, dev, mb, W, graph):
    from ddrl_b200.config import PPOConfig
    from ddrl_b200.learner import FCNetLearner
    L = FCNetLearner(pr["P"], pr["D"], pr["A"], PPOConfig(num_sgd_iter=ME, sgd_minibatch_size=mb), dev,
                     theta=torch.from_numpy(pr["theta0"]), use_graph=graph, filter_mode="stream", filter_workers=W)
    _set_filter(L, pr["filt0"])
    return L


def _multi_worker(rank, world, port, q):
    try:
        import torch.distributed as dist
        from tests.test_gpu_multi import _teardown
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
        torch.cuda.set_device(rank)
        dev = torch.device("cuda", rank)
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
        pr = _problem("FullyDecentral", MT, MC, 21)
        Cl = MC // world
        sl = slice(rank * Cl, (rank + 1) * Cl)
        to = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
        rng = np.random.default_rng(1)
        perms = np.stack([np.stack([rng.permutation(MNB) for _ in range(ME)]) for _ in range(pr["P"])]).astype(np.int32)
        L = _multi_learner(pr, dev, (MT * MC) // MNB, MW, True)
        args = (to(pr["raw"][:, :, sl]), to(pr["boot"][:, sl]), to(pr["rewards"][:, :, sl]), to(pr["dones"][:, sl]),
                to(pr["eps"][:, :, sl]), to(perms))
        for _ in range(3):
            L.learn_on_rollout(*args)
        torch.cuda.synchronize()
        res = (L.theta.cpu().numpy(), L.filt_n.cpu().numpy(), L.filt_M.cpu().numpy(), L.filt_S.cpu().numpy())
        gathered = [None] * world
        dist.all_gather_object(gathered, res)
        if rank == 0:
            same = all(all(np.array_equal(a, b) for a, b in zip(g, res)) for g in gathered)
            q.put(res + (same,))
            time.sleep(1.0)
        _teardown(L, dist)
    except Exception as exc:
        import traceback
        q.put(("error", rank, "".join(traceback.format_exception(exc))))
        raise


def test_world_2_stream_mode_equals_one_gpu_with_twice_the_workers():
    """2 ranks x 2 workers on half the envs each == 1 GPU x 4 workers on all envs: the filter state bit for bit (the same
    stream partials, folded in the same order), the weights within the reduction-order tolerance of the batch-mode test."""
    import torch.multiprocessing as mp
    world = 2
    if torch.cuda.device_count() < world:
        pytest.skip("needs 2 GPUs")
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_multi_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = q.get(timeout=300)
    if isinstance(res[0], str) and res[0] == "error":
        for p in procs:
            p.join(timeout=30)
            if p.is_alive():
                p.terminate()
        pytest.fail(f"rank {res[1]} failed:\n{res[2]}")
    th2, n2, M2, S2, same = res
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert same, "ranks diverged"
    pr = _problem("FullyDecentral", MT, MC, 21)
    rng = np.random.default_rng(1)
    perms = np.stack([np.stack([rng.permutation(MNB) for _ in range(ME)]) for _ in range(pr["P"])]).astype(np.int32)
    Cl, MBl = MC // world, (MT * MC) // MNB // world
    order = []
    for b in range(MNB):
        for r in range(world):
            for j in range(MBl):
                t, cl = divmod(b * MBl + j, Cl)
                order.append(t * MC + r * Cl + cl)
    shuffle = np.tile(np.asarray(order, dtype=np.int32), (pr["P"], 1))
    L = _multi_learner(pr, "cuda", (MT * MC) // MNB, MW * world, False)
    for _ in range(3):
        L.learn_on_rollout(_dev(pr["raw"]), _dev(pr["boot"]), _dev(pr["rewards"]), _dev(pr["dones"]), _dev(pr["eps"]),
                           _dev(perms), _dev(shuffle))
    torch.cuda.synchronize()
    assert np.array_equal(L.filt_n.cpu().numpy(), n2)
    assert np.array_equal(L.filt_M.cpu().numpy(), M2) and np.array_equal(L.filt_S.cpu().numpy(), S2)
    th1 = L.theta.cpu().numpy()
    for p in range(pr["P"]):
        assert scaled_err(th2[p], th1[p]) < 1e-4
        assert scaled_err(th2[p].astype(np.float64) - pr["theta0"][p], th1[p].astype(np.float64) - pr["theta0"][p]) < 2e-3

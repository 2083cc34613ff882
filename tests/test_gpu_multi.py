"""GPU (needs >= 2 devices; run with `gpurun --gpus 2`): the 2-rank NCCL data-parallel learner reproduces the
1-GPU result on the same global batch (shard by env, gradient all-reduce per optimizer step, rank-ordered filter
merge, advantage-moment all-reduce)."""
import os
import socket
import time

import numpy as np
import pytest
import torch

from tests.util import ckpt_theta, scaled_err, synth_obs

pytestmark = pytest.mark.gpu

T, C, E, NB = 16, 64, 2, 4
ITERS = 3      # learner iterations per run: the second one captures the preparation phase into a CUDA graph, the third replays it
ARCH = "FullyDecentral"
UPD_TOL = 2e-3     # measured on hardware: 5e-5 (world 2); was 0.2 before the test had ever run


def _problem():
    theta, filt, D, A = ckpt_theta(ARCH)
    P = theta.shape[0]
    rng = np.random.default_rng(5)
    raw = synth_obs(filt, T * C, 1).reshape(P, T, C, D)
    boot = synth_obs(filt, C, 2)
    rewards = (0.3 + 0.5 * rng.standard_normal((P, T, C))).astype(np.float32)
    dones = (rng.random((T, C)) < 0.05).astype(np.uint8)
    eps = rng.standard_normal((P, T, C, A)).astype(np.float32)
    perms = np.stack([np.stack([rng.permutation(NB) for _ in range(E)]) for _ in range(P)]).astype(np.int32)
    return dict(theta=theta, filt=filt, D=D, A=A, P=P, raw=raw, boot=boot, rewards=rewards, dones=dones, eps=eps, perms=perms)


def _learner(pr, dev, mb, mode="fp32", fuse=True, graph=False):
    from ddrl_b200.config import PPOConfig
    from ddrl_b200.learner import FCNetLearner
    cfg = PPOConfig(num_sgd_iter=E, sgd_minibatch_size=mb)
    L = FCNetLearner(pr["P"], pr["D"], pr["A"], cfg, dev, theta=torch.from_numpy(pr["theta"]), use_graph=graph, mode=mode,
                     fuse_tail=fuse)
    filt = [(1000, M, S * (999.0 / (n - 1))) for n, M, S in pr["filt"]]
    L.filt_n.copy_(torch.tensor([f[0] for f in filt]))
    L.filt_M.copy_(torch.from_numpy(np.stack([f[1] for f in filt])))
    L.filt_S.copy_(torch.from_numpy(np.stack([f[2] for f in filt])))
    return L


def _teardown(L, dist):
    """Release captured graphs (they hold NCCL work) before the communicator goes away, and never let the teardown hang the
    test: the result is already in the queue."""
    import threading
    L._graph = None
    if getattr(L, "_prep_graphs", None):
        L._prep_graphs = {}
    torch.cuda.synchronize()
    dist.barrier()
    t = threading.Thread(target=dist.destroy_process_group, daemon=True)
    t.start()
    t.join(timeout=15.0)
    os._exit(0)


def _worker(rank, world, port, q, mode, fuse, graph):
    try:
        _worker_body(rank, world, port, q, mode, fuse, graph)
    except Exception as exc:  # surface the failure instead of leaving the parent waiting on the queue
        import traceback
        q.put(("error", rank, "".join(traceback.format_exception(exc))))
        raise


def _worker_body(rank, world, port, q, mode, fuse, graph):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    pr = _problem()
    Cl = C // world
    sl = slice(rank * Cl, (rank + 1) * Cl)
    to = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    L = _learner(pr, dev, (T * C) // NB, mode, fuse, graph)
    args = (to(pr["raw"][:, :, sl]), to(pr["boot"][:, sl]), to(pr["rewards"][:, :, sl]), to(pr["dones"][:, sl]),
            to(pr["eps"][:, :, sl]), to(pr["perms"]))
    for _ in range(ITERS):
        stats = L.learn_on_rollout(*args)
    if graph:
        assert L._prep_graphs, f"the preparation phase was not captured at world {world}: {getattr(L, 'graph_error', None)}"
    assert (L._peers is not None) == fuse, "fused tail must use the peer exchange, the 3-kernel path NCCL"
    torch.cuda.synchronize()
    th = L.theta.cpu().numpy()
    gathered = [None] * world
    dist.all_gather_object(gathered, th)
    if rank == 0:
        q.put((th, stats, L.filt_n.cpu().numpy(), L.filt_M.cpu().numpy(), [np.array_equal(g, th) for g in gathered]))
        time.sleep(1.0)      # let the queue's feeder thread flush before os._exit
    _teardown(L, dist)


@pytest.mark.parametrize("world", [2, 4, 8])
@pytest.mark.parametrize("mode,fuse,graph", [("fp32", True, False), ("fp32", False, False), ("tc", True, True)],
                         ids=["fp32-peer", "fp32-nccl", "tc-peer-persistent"])
def test_multi_gpu_learner_equals_one_gpu_learner(mode, fuse, graph, world):
    """SURVEY.md §8-e: the G-GPU run equals the 1-GPU run on the same global batch.
    fuse=True: ONE kernel per step with the in-kernel NVLink all-reduce (csrc/sgd_tail.cuh); fuse=False: NCCL."""
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q, mode, fuse, graph)) for r in range(world)]
    for p in procs:
        p.start()
    res = q.get(timeout=300)
    if isinstance(res[0], str) and res[0] == "error":
        for p in procs:
            p.join(timeout=30)
            if p.is_alive():
                p.terminate()
        pytest.fail(f"rank {res[1]} failed:\n{res[2]}")
    th2, stats2, n2, M2, same = res
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert all(same), "ranks diverged: replicated weights must stay bit-identical"

    # 1-GPU run on the full batch, rows ordered so every minibatch is the union of the ranks' local minibatches
    pr = _problem()
    Cl, MBl = C // world, (T * C) // NB // world
    order = []
    for b in range(NB):
        for r in range(world):
            for j in range(MBl):
                t, cl = divmod(b * MBl + j, Cl)
                order.append(t * C + r * Cl + cl)
    shuffle = np.tile(np.asarray(order, dtype=np.int32), (pr["P"], 1))
    dev = torch.device("cuda", 0)
    to = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    L = _learner(pr, dev, (T * C) // NB, mode)
    args1 = (to(pr["raw"]), to(pr["boot"]), to(pr["rewards"]), to(pr["dones"]), to(pr["eps"]), to(pr["perms"]), to(shuffle))
    for _ in range(ITERS):
        stats1 = L.learn_on_rollout(*args1)
    torch.cuda.synchronize()
    assert np.array_equal(L.filt_n.cpu().numpy(), n2)
    np.testing.assert_allclose(M2, L.filt_M.cpu().numpy(), rtol=1e-12, atol=1e-13)
    th1 = L.theta.cpu().numpy()
    for p in range(pr["P"]):
        upd1 = th1[p].astype(np.float64) - pr["theta"][p]
        upd2 = th2[p].astype(np.float64) - pr["theta"][p]
        e_th, e_upd = scaled_err(th2[p], th1[p]), scaled_err(upd2, upd1)
        if os.environ.get("DDRL_ERRLOG"):
            with open(os.environ["DDRL_ERRLOG"], "a") as f:
                f.write(f"multi world={world} mode={mode} fuse={fuse} p={p} theta_err={e_th:.3e} update_err={e_upd:.3e}\n")
        assert e_th < 1e-4
        assert e_upd < UPD_TOL          # FP32 reduction order differs; Adam amplifies (see DESIGN.md §2)
        for k in ("total_loss", "policy_loss", "vf_loss", "kl", "entropy"):
            assert abs(stats2[p][k] - stats1[p][k]) < 1e-4 * max(1.0, abs(stats1[p][k])), (k, stats2[p][k], stats1[p][k])


# ---- shared GraphNet policy: the tensor-core step with the in-kernel all-reduce (csrc/graphnet_tc.cu + sgd_tail.cuh) ----------
GT, GN_ENVS, GE, GNB = 8, 32, 2, 4
GC = GN_ENVS * 4


def _gn_problem():
    from tests.test_gpu_graphnet import _inputs, _theta
    A = 2
    R = GT * GC
    idx, state, adj = _inputs(R, 41, "ring")
    idx = np.tile(np.arange(4, dtype=np.int32), R // 4)
    bidx, bstate, badj = _inputs(GC, 42, "ring")
    bidx = np.tile(np.arange(4, dtype=np.int32), GC // 4)
    rng = np.random.default_rng(43)
    rewards = (0.3 + 0.5 * rng.standard_normal((GT, GC))).astype(np.float32)
    dones = (rng.random((GT, GN_ENVS)) < 0.05).astype(np.uint8)
    eps = rng.standard_normal((GT, GC, A)).astype(np.float32)
    perms = np.stack([rng.permutation(GNB) for _ in range(GE)]).astype(np.int32)
    return dict(A=A, idx=idx.reshape(GT, GC), state=state.reshape(GT, GC, 4, 23), adj=adj.reshape(GT, GC, 4, 4), bidx=bidx,
                bstate=bstate, badj=badj, rewards=rewards, dones=dones, eps=eps, perms=perms, theta=_theta(A, 5, big=True).float())


def _gn_worker(rank, world, port, q):
    try:
        import torch.distributed as dist
        from ddrl_b200.config import PPOConfig
        from ddrl_b200.learner import GraphNetLearner
        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
        torch.cuda.set_device(rank)
        dev = torch.device("cuda", rank)
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
        pr = _gn_problem()
        Cl, Nl = GC // world, GN_ENVS // world
        sl, sn = slice(rank * Cl, (rank + 1) * Cl), slice(rank * Nl, (rank + 1) * Nl)
        to = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
        cfg = PPOConfig(num_sgd_iter=GE, sgd_minibatch_size=(GT * GC) // GNB)
        L = GraphNetLearner(pr["A"], cfg, dev, theta=pr["theta"].reshape(1, -1), step="tc")
        stats = L.learn_on_rollout(to(pr["idx"][:, sl]), to(pr["state"][:, sl]), to(pr["adj"][:, sl]), to(pr["bidx"][sl]),
                                   to(pr["bstate"][sl]), to(pr["badj"][sl]), to(pr["rewards"][:, sl]), to(pr["dones"][:, sn]),
                                   to(pr["eps"][:, sl]), to(pr["perms"]))
        assert L._peers is not None, "the GraphNet tensor-core step must use the peer exchange at world > 1"
        torch.cuda.synchronize()
        th = L.theta.cpu().numpy()
        gathered = [None] * world
        dist.all_gather_object(gathered, th)
        if rank == 0:
            q.put((th, stats, [np.array_equal(g, th) for g in gathered]))
            time.sleep(1.0)      # let the queue's feeder thread flush before os._exit
        _teardown(L, dist)
    except Exception as exc:
        import traceback
        q.put(("error", rank, "".join(traceback.format_exception(exc))))
        raise


@pytest.mark.parametrize("world", [2, 8])
def test_multi_gpu_graphnet_learner_equals_one_gpu_learner(world):
    """The shared GraphNet policy trained by `world` ranks (rollout sharded by env, gradient all-reduce inside the persistent
    tensor-core step kernel) equals the 1-GPU run on the same global batch; replicated weights stay bit-identical."""
    import torch.multiprocessing as mp
    from ddrl_b200.config import PPOConfig
    from ddrl_b200.learner import GraphNetLearner
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_gn_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = q.get(timeout=300)
    if isinstance(res[0], str) and res[0] == "error":
        for p in procs:
            p.join(timeout=30)
            if p.is_alive():
                p.terminate()
        pytest.fail(f"rank {res[1]} failed:\n{res[2]}")
    th2, stats2, same = res
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert all(same), "ranks diverged: replicated weights must stay bit-identical"
    pr = _gn_problem()
    Cl, MBl = GC // world, (GT * GC) // GNB // world
    order = []
    for b in range(GNB):
        for r in range(world):
            for j in range(MBl):
                t, cl = divmod(b * MBl + j, Cl)
                order.append(t * GC + r * Cl + cl)
    dev = torch.device("cuda", 0)
    to = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    cfg = PPOConfig(num_sgd_iter=GE, sgd_minibatch_size=(GT * GC) // GNB)
    L = GraphNetLearner(pr["A"], cfg, dev, theta=pr["theta"].reshape(1, -1), step="tc")
    stats1 = L.learn_on_rollout(to(pr["idx"]), to(pr["state"]), to(pr["adj"]), to(pr["bidx"]), to(pr["bstate"]), to(pr["badj"]),
                                to(pr["rewards"]), to(pr["dones"]), to(pr["eps"]), to(pr["perms"]),
                                to(np.asarray(order, dtype=np.int32)))
    torch.cuda.synchronize()
    th1 = L.theta.cpu().numpy().reshape(-1)
    th0 = pr["theta"].numpy().astype(np.float64)
    e_upd = scaled_err(th2.reshape(-1).astype(np.float64) - th0, th1.astype(np.float64) - th0)
    if os.environ.get("DDRL_ERRLOG"):
        with open(os.environ["DDRL_ERRLOG"], "a") as f:
            f.write(f"multi graphnet world={world} update_err={e_upd:.3e}\n")
    assert e_upd < UPD_TOL
    for k in ("total_loss", "policy_loss", "vf_loss", "kl", "entropy"):
        assert abs(stats2[0][k] - stats1[0][k]) < 1e-4 * max(1.0, abs(stats1[0][k])), (k, stats2[0][k], stats1[0][k])

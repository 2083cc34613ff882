"""CPU: the schedule of ddrl_filter_stream (csrc/filter_stream.cu) transcribed in numpy float64 — chunk Welford partials,
the fixed-order scan of the chunk partials over 32 groups seeded with the running state, the re-walk of every chunk from
its prefix state — against RLlib's row-by-row sampler filtering (tests/filter_stream_oracle.py), for every chunk size."""
import numpy as np
import pytest

from tests.filter_stream_oracle import filter_stream, running_stat, state_error_bound, stream_rows

GROUPS = 32      # FS_GROUPS of the kernel


def _push(s, x):
    """RunningStat.push in the kernel's operation order."""
    n1 = s[0]
    n = n1 + 1.0
    if n1 == 0.0:
        return (n, x.copy(), s[2].copy())
    delta = x - s[1]
    return (n, s[1] + delta / n, s[2] + delta * delta * n1 / n)


def _merge(a, b):
    """RunningStat.update; an empty side leaves the other unchanged."""
    if b[0] == 0.0:
        return a
    if a[0] == 0.0:
        return b
    n = a[0] + b[0]
    delta = a[1] - b[1]
    return (n, (a[0] * a[1] + b[0] * b[1]) / n, a[2] + b[2] + delta * delta * a[0] * b[0] / n)


def kernel_schedule(x, T, C, W, start, clip, chunk):
    """-> (y [T*C, D] float64 before the float32 rounding, parts [W] of (count, mean, M2))."""
    x = np.asarray(x, dtype=np.float64)
    D = x.shape[1]
    empty = (0.0, np.zeros(D), np.zeros(D))
    run = (float(start[0]), np.asarray(start[1], np.float64), np.asarray(start[2], np.float64))
    y = np.empty_like(x)
    parts = []
    for rows in stream_rows(T, C, W):
        L = len(rows)
        nch = -(-L // chunk)
        chunks = [rows[k * chunk:(k + 1) * chunk] for k in range(nch)]
        # 1. chunk partials from an empty state
        part = []
        for ch in chunks:
            s = empty
            for r in ch:
                s = _push(s, x[r])
            part.append(s)
        # 2. scan: group totals, exclusive prefix of every group on the running state, the stream's buffer, chunk prefixes
        G = -(-nch // GROUPS)
        groups = [range(min(l * G, nch), min(l * G + G, nch)) for l in range(GROUPS)]
        tot = []
        for g in groups:
            s = empty
            for k in g:
                s = _merge(s, part[k])
            tot.append(s)
        buf = empty
        for t_ in tot:
            buf = _merge(buf, t_)
        parts.append(buf)
        prefix = [None] * nch
        for l, g in enumerate(groups):
            pre = run
            for t_ in tot[:l]:
                pre = _merge(pre, t_)
            for k in g:
                prefix[k] = pre
                pre = _merge(pre, part[k])
        # 3. re-walk every chunk from its prefix state
        for k, ch in enumerate(chunks):
            s = prefix[k]
            for r in ch:
                s = _push(s, x[r])
                var = s[2] / (s[0] - 1.0) if s[0] > 1.0 else s[1] * s[1]
                v = (x[r] - s[1]) / (np.sqrt(var) + 1e-8)
                y[r] = np.clip(v, -clip, clip) if clip else v
    return y, parts


def _rollout(T, C, D, seed, scale=3.0):
    rng = np.random.default_rng(seed)
    return (rng.standard_normal(D) * scale + rng.standard_normal((T * C, D)) * rng.uniform(0.5, 2.0, D)).astype(np.float32)


START = {"empty": lambda D, rng: (0, np.zeros(D), np.zeros(D)),
         "small": lambda D, rng: (3, rng.standard_normal(D), rng.uniform(0.5, 2.0, D)),
         "warm": lambda D, rng: (20_000_000, rng.standard_normal(D), rng.uniform(0.5, 2.0, D) * 2e7)}


@pytest.mark.parametrize("start", sorted(START))
@pytest.mark.parametrize("chunk", [1, 2, 3, 5, 7, 8, 13, 64, 1000])
@pytest.mark.parametrize("T,C,W", [(5, 6, 1), (5, 6, 2), (7, 12, 3), (3, 8, 8), (40, 4, 2)])
def test_schedule_equals_row_by_row_filter(T, C, W, chunk, start):
    """Chunks that straddle steps (chunk not a multiple of C/W) and streams of one column; clip on and off."""
    D = 5
    rng = np.random.default_rng(T * 100 + C * 10 + W)
    st = START[start](D, rng)
    x = _rollout(T, C, D, T + C + W)
    for clip in (None, 1.5):
        y_ref, drv, bufs, mean, std = filter_stream(x, T, C, W, st, clip, row_state=True)
        y, parts = kernel_schedule(x, T, C, W, st, clip, chunk)
        Cw = C // W
        # the first chunk of every stream is walked from the running state itself: bit for bit
        for rows in stream_rows(T, C, W):
            first = rows[:chunk]
            np.testing.assert_array_equal(y[first], y_ref[first])
        err = np.abs(y - y_ref) / state_error_bound(x, mean, std, 1e-12)
        assert err.max() <= 1.0, (Cw, err.max())
        for p, b in zip(parts, bufs):
            assert p[0] == b.n
            np.testing.assert_allclose(p[1], b.mean, rtol=1e-12, atol=1e-12 * np.abs(b.mean).max())
            np.testing.assert_allclose(p[2], b._S, rtol=1e-12, atol=1e-300)
        # the parts folded into the start state in worker order == the synchronised driver filter
        run = running_stat(*st)
        for p in parts:
            run.update(running_stat(int(p[0]), p[1], p[2]))
        assert run.n == drv.n
        np.testing.assert_allclose(run.mean, drv.mean, rtol=1e-12, atol=1e-12 * np.abs(drv.mean).max())
        np.testing.assert_allclose(run._S, drv._S, rtol=1e-12)


def test_worker_split_and_row_order_on_a_hand_written_rollout():
    """T = 2 steps, C = 4 columns (2 envs x 2 agent columns), W = 2 workers: worker 0 owns env 0 (columns 0, 1), worker 1
    env 1; each filters its rows step-major.  From an empty filter the first row of every worker maps to 0."""
    assert stream_rows(2, 4, 2) == [[0, 1, 4, 5], [2, 3, 6, 7]]
    assert stream_rows(2, 4, 1) == [[0, 1, 2, 3, 4, 5, 6, 7]]
    x = np.array([[1.0], [3.0], [10.0], [20.0], [5.0], [7.0], [40.0], [0.0]])
    y, drv, bufs = filter_stream(x, 2, 4, 2, (0, np.zeros(1), np.zeros(1)))
    # worker 0 sees 1, 3, 5, 7 ; worker 1 sees 10, 20, 40, 0
    assert y[0, 0] == 0.0 and y[2, 0] == 0.0
    assert y[1, 0] == (3.0 - 2.0) / (np.sqrt(2.0) + 1e-8)              # mean 2, S = 2 after two pushes
    assert y[4, 0] == (5.0 - 3.0) / (np.sqrt(4.0) + 1e-8)              # mean 3, S = 8, n = 3
    assert y[3, 0] == (20.0 - 15.0) / (np.sqrt(50.0) + 1e-8)
    assert [b.n for b in bufs] == [4, 4] and drv.n == 8
    assert bufs[0].mean[0] == 4.0 and bufs[1].mean[0] == 17.5
    yk, _ = kernel_schedule(x, 2, 4, 2, (0, np.zeros(1), np.zeros(1)), None, 3)
    np.testing.assert_allclose(yk, y, rtol=1e-15)

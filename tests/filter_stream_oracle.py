"""RLlib's row-by-row observation filtering on the sampler side, restated on the oracle's RunningStat / MeanStdFilter
(oracle/ddrl_oracle.py, a4).  Test infrastructure only.

RLlib 1.0.1 (evaluation/sampler.py _process_observations) calls a policy's MeanStdFilter once per observation row: the
unvectorised __call__ pushes the row into `rs` and `buffer` and normalises it with the updated state.  Every rollout
worker holds its own copy of the driver's filter from the start of the iteration; FilterManager.synchronize then applies
the workers' buffers to the driver copy in worker order (apply_changes -> RunningStat.update)."""
import copy
from typing import List, Tuple

import numpy as np

from oracle.ddrl_oracle import MeanStdFilter, RunningStat


def stream_rows(T: int, C: int, W: int) -> List[List[int]]:
    """Rows of a [T, C] rollout (row t*C + c) that worker w filters, in its order: columns [w*C/W, (w+1)*C/W), step-major."""
    if C % W:
        raise ValueError(f"C={C} columns do not split into W={W} workers")
    Cw = C // W
    return [[t * C + w * Cw + c for t in range(T) for c in range(Cw)] for w in range(W)]


def running_stat(n: int, M, S) -> RunningStat:
    """A RunningStat holding (n, M, S)."""
    rs = RunningStat(np.asarray(M).shape)
    rs._n, rs._M, rs._S = int(n), np.array(M, dtype=np.float64), np.array(S, dtype=np.float64)
    return rs


def filter_stream(x: np.ndarray, T: int, C: int, W: int, start: Tuple[int, np.ndarray, np.ndarray], clip=None,
                  row_state: bool = False):
    """x [T*C, D] raw rows; start = (n, M, S) the driver filter.  One filter copy per worker starts from `start`, its rows
    are called one at a time in (t, c) order, then the buffers are applied to the driver in worker order.
    -> (y [T*C, D] float64 normalised rows, driver RunningStat after the synchronisation, worker buffers); with
    row_state also (mean [T*C, D], std [T*C, D]): the statistics each row was normalised with."""
    x = np.asarray(x, dtype=np.float64)
    D = x.shape[1]
    driver = running_stat(*start)
    y = np.empty_like(x)
    mean, std = np.empty_like(x), np.empty_like(x)
    bufs = []
    for rows in stream_rows(T, C, W):
        f = MeanStdFilter((D,), clip=clip)
        f.rs = copy.deepcopy(driver)
        for r in rows:
            y[r] = f(x[r])
            mean[r], std[r] = f.rs.mean, f.rs.std
        bufs.append(f.buffer)
    for b in bufs:
        driver.update(b)
    return (y, driver, bufs, mean, std) if row_state else (y, driver, bufs)


class StreamFilter:
    """Stands in for `PolicyState.filt` in `fcnet_learner_iteration`: the updating call filters a [T*C, D] rollout worker
    by worker and row by row (`filter_stream`); a call with update=False normalises with the current state, unpushed."""

    def __init__(self, D: int, start, T: int, C: int, W: int, clip=None):
        self.filt = MeanStdFilter((D,), clip=clip)
        self.filt.rs = running_stat(*start)
        self.T, self.C, self.W = T, C, W

    @property
    def rs(self) -> RunningStat:
        return self.filt.rs

    def __call__(self, x, update=True):
        if not update:
            return self.filt(x, update=False)
        rs = self.filt.rs
        y, self.filt.rs, _ = filter_stream(x, self.T, self.C, self.W, (rs._n, rs._M, rs._S), self.filt.clip)
        return y


def state_error_bound(x, mean, std, rel: float = 1e-10):
    """How far a normalised row may move when its state (mean, std) carries a relative error of ~1e-12: the error is carried
    through the subtraction and the division, rel * (|x| + |mean|) / (std + 1e-8)."""
    return rel * (np.abs(np.asarray(x, np.float64)) + np.abs(mean)) / (std + 1e-8)

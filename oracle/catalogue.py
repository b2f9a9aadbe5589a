"""TEST INFRASTRUCTURE ONLY -- the oracle of the posterior of a catalogue of mixed planet counts
(``bnn_summarize_instability_ragged``, ``bnn_survival_instability_ragged``, ``MultiSWAG.posterior_summary`` with
per-system trio counts).

System n owns rows off[n] .. off[n+1] - 1 of the system-major arrays, off = [0, cumsum(counts)].  Its min over trios is
taken the way the kernels take it, so the result can feed ``restatement.posterior_stats`` unchanged:
  * the sampled time: fmin from +inf (a unit whose trio draws are all NaN is +inf);
  * mu* and its std: the first trio's (mu, std), replaced by a later trio's only when its mu is strictly smaller (a NaN
    mu is never smaller), then a NaN mu* or std* is +inf (the kernels rank NaN predictions last).
"""
from __future__ import annotations

import numpy as np

from . import restatement


def offsets(counts) -> np.ndarray:
    c = np.asarray(counts, np.int64).reshape(-1)
    return np.concatenate([[0], np.cumsum(c)]).astype(np.int64)


def ragged_min_time(t, counts) -> np.ndarray:
    """t [R, U] -> [N, U] float32: per system, fmin over its trio rows from +inf."""
    t = np.asarray(t, np.float32)
    off = offsets(counts)
    tmin = np.fmin.reduceat(t, off[:-1], axis=0)   # NaN only where every trio is NaN
    return np.where(np.isnan(tmin), np.float32(np.inf), tmin).astype(np.float32)


def ragged_min_pred(pred, counts):
    """pred [R, U, 2] -> (mu* [N, U], std* [N, U]) float32: the (mu, std) of the trio of smallest mu, first trio on ties
    and NaN, NaN mapped to +inf."""
    pred = np.asarray(pred, np.float32)
    off = offsets(counts)
    N = off.size - 1
    best = pred[off[:-1]].copy()   # [N, U, 2]: the first trio
    for k in range(1, int(np.diff(off).max())):
        has = off[:-1] + k < off[1:]
        rows = pred[np.minimum(off[:-1] + k, off[-1] - 1)]
        take = has[:, None] & (rows[..., 0] < best[..., 0])
        best[take] = rows[take]
    mu, sd = best[..., 0], best[..., 1]
    inf = np.float32(np.inf)
    return np.where(np.isnan(mu), inf, mu), np.where(np.isnan(sd), inf, sd)


def catalogue_stats(t, pred, counts):
    """``restatement.posterior_stats`` of a catalogue: t [R, U], pred [R, U, 2], counts [N] -> per-system dict, the min
    over each system's trios taken by ``ragged_min_time`` / ``ragged_min_pred`` and handed over as one trio."""
    tmin = ragged_min_time(t, counts)
    mu, sd = ragged_min_pred(pred, counts)
    return restatement.posterior_stats(tmin.T[:, :, None], np.stack([mu, sd], -1).transpose(1, 0, 2)[:, :, None, :])


def catalogue_survival(t, thresholds, counts) -> np.ndarray:
    """``survival.survival_fraction`` of a catalogue: t [R, U] sampled log10 instability times, thresholds [J], counts [N]
    -> [N, J] float32: #{u : ragged_min_time(t)[n, u] > thresholds[j]} / U, counted exactly, divided by U in float64 and
    rounded to fp32 once."""
    thr = np.asarray(thresholds, np.float32).reshape(-1)
    tmin = ragged_min_time(t, counts)
    count = np.stack([(tmin > v).sum(1) for v in thr], 1)
    return (count.astype(np.float64) / tmin.shape[1]).astype(np.float32)

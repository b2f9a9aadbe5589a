"""TEST INFRASTRUCTURE ONLY -- the oracle of the survival probability (``bnn_survival_instability``,
``MultiSWAG.posterior_survival``).

Counts the sampled instability times the way the reference's figure scripts compute everything, from the samples: the min
over trios (as ``bnn_summarize_instability`` takes it, fmin from +inf, so an all-NaN unit is +inf), compared strictly with
each threshold in fp32, counted exactly, divided by U in float64 and rounded to fp32 once.
"""
from __future__ import annotations

import numpy as np


def survival_fraction(t, thresholds, n_trios: int = 1) -> np.ndarray:
    """t [N*n_trios, U] sampled log10 instability times (row = system*n_trios + trio), thresholds [J] ->
    [N, J] float32: #{u : min_r t[n*n_trios + r, u] > thresholds[j]} / U."""
    t = np.asarray(t, np.float32)
    thr = np.asarray(thresholds, np.float32).reshape(-1)
    rows, U = t.shape
    N = rows // n_trios
    tr = t.reshape(N, n_trios, U)
    tmin = np.full((N, U), np.inf, np.float32)
    for r in range(n_trios):
        tmin = np.fmin(tmin, tr[:, r])
    count = np.stack([(tmin > v).sum(1) for v in thr], 1)
    return (count.astype(np.float64) / U).astype(np.float32)

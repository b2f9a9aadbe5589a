"""TEST INFRASTRUCTURE ONLY -- the oracle of the variance decomposition (``bnn_decompose_uncertainty``,
``MultiSWAG.posterior_uncertainty``).

Per prediction row, in numpy float64, two-pass: the model means first, then the deviations from them.  Unit u = k*S + s
is sample s of model k.  Population (ddof = 0) moments of the untruncated per-unit normals, rounded to fp32 once.
"""
from __future__ import annotations

import numpy as np


def variance_decomposition(pred, units_per_model: int) -> np.ndarray:
    """pred [rows, U, 2] of (mu, sigma) -> [rows, 5] float32: mean_mu, aleatoric = mean sigma^2, epistemic = between +
    within, between_models = (1/M) sum_k (m_k - mean)^2, within_models = (1/M) sum_k (1/S) sum_s (mu_ks - m_k)^2.
    A non-finite mu makes every column but aleatoric NaN; a non-finite sigma makes aleatoric NaN."""
    pred = np.asarray(pred, np.float32)
    rows, U, _ = pred.shape
    S = int(units_per_model)
    mu = pred[:, :, 0].astype(np.float64).reshape(rows, U // S, S)
    sd = pred[:, :, 1].astype(np.float64)
    with np.errstate(invalid="ignore", over="ignore"):
        m = mu.mean(2)                                    # [rows, M]
        mean = m.mean(1)                                  # [rows]
        between = ((m - mean[:, None]) ** 2).mean(1)
        within = ((mu - m[:, :, None]) ** 2).mean(2).mean(1)
        aleatoric = (sd * sd).mean(1)
    out = np.stack([mean, aleatoric, between + within, between, within], 1)
    out[np.ix_(~np.isfinite(pred[:, :, 0]).all(1), [0, 2, 3, 4])] = np.nan
    out[~np.isfinite(pred[:, :, 1]).all(1), 1] = np.nan
    return out.astype(np.float32)


def epistemic_direct(pred) -> np.ndarray:
    """pred [rows, U, 2] -> float64 [rows]: (1/U) sum_u (mu_u - mean)^2 in one step, which equals between + within in
    real arithmetic (the law of total variance over the equal-size models)."""
    mu = np.asarray(pred, np.float32)[:, :, 0].astype(np.float64)
    with np.errstate(invalid="ignore", over="ignore"):
        return ((mu - mu.mean(1, keepdims=True)) ** 2).mean(1)

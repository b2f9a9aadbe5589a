"""TEST INFRASTRUCTURE ONLY -- the oracle of the posterior attribution (``bnn_posterior_saliency``,
``MultiSWAG.posterior_attribution``).

For each unit's flat weights and explicit summary draws, torch autograd on the restatement gives mu_u and
g_u = d mu_u / d x of the masked input (the way feature_importance.py's gradforward differentiates, and the way
tests/test_gpu_train.py checks bnn_saliency); the reduction over units and time steps runs in numpy float64.
"""
from __future__ import annotations

import numpy as np
import torch

from . import restatement as R


def unit_gradients(spec: R.ModelSpec, thetas, x, eps):
    """thetas [U, d] flat weights, x [rows, T, F], eps [U, rows, 2L] (eps1 | eps2) -> (g [U, rows, T, F] float32,
    mu [U, rows] float32): each unit's predicted mean and its gradient with respect to the masked input."""
    thetas, x, eps = (torch.as_tensor(np.asarray(a, np.float32)) for a in (thetas, x, eps))
    L = eps.shape[2] // 2
    gs, mus = [], []
    for u in range(thetas.shape[0]):
        p = R.unflatten(spec, thetas[u])
        xz = R.zero_columns(spec, x).clone().requires_grad_(True)
        s = R.compute_summary_stats(spec, p, xz, eps[u, :, :L], eps[u, :, L:])
        mu, _ = R.predict_instability(spec, p, s)
        (g,) = torch.autograd.grad(mu.sum(), xz)
        gs.append(g.numpy())
        mus.append(mu.detach().reshape(-1).numpy())
    return np.stack(gs), np.stack(mus)


def reduce_attribution(g, mu):
    """g [U, rows, T, F], mu [U, rows] -> float64 (attribution [rows, 2, F], mu_mean [rows], abs_shift [rows, F]):
    importance = (1/U) sum_u (1/T) sum_t g^2, shift = (1/U) sum_u sum_t g, mu_mean = (1/U) sum_u mu, and
    abs_shift = (1/U) sum_u sum_t |g|, the scale a shift's rounding error is measured against."""
    g = np.asarray(g, np.float64)
    U, T = g.shape[0], g.shape[2]
    importance = (g * g).sum(2).sum(0) / (U * T)
    shift = g.sum(2).sum(0) / U
    return (np.stack([importance, shift], 1), np.asarray(mu, np.float64).mean(0), np.abs(g).sum(2).sum(0) / U)

"""Posterior post-processing on the GPU (SURVEY.md section 8f, rank 1).

Replaces the host-side numpy tail of the reference's evaluation scripts -- ``fast_truncnorm`` (left = 4),
resampling of draws >= 9 from the analytic prior, min over trios, per-system median / percentiles
(figures/main_figures.py:167-277, figures/multiswag_5_planet.py:306-481) -- so that only ``[N, 8]`` leaves the
device instead of the ``[N, U, 2]`` prediction block.  ``survival`` counts the same sampled times against thresholds:
P(T_inst > t) per system.  ``uncertainty`` splits each row's predictive variance into aleatoric, between-model and
within-model parts.
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import _lib

STAT_NAMES = ("average", "median", "l", "u", "ll", "uu", "median_mu", "median_std")  # multiswag_5_planet.py:476-481


def sample_instability(pred: torch.Tensor, seed: int = 0, row_offset: int = 0, left: float = 4.0, nsamp: int = 40):
    """pred [rows, U, 2] (system-major (mu, std)) -> sampled log10 instability times [rows, U]."""
    lib = _lib.load()
    _lib.require_cuda(pred, "pred")
    pred = pred.contiguous().float()
    rows, U = pred.shape[0], pred.shape[1]
    t = torch.empty((rows, U), device=pred.device, dtype=torch.float32)
    if rows == 0:
        return t
    with torch.cuda.device(pred.device), _lib.nvtx("bnn:K7 sample_instability"):
        _lib.check(lib.bnn_sample_instability(_lib.ptr(pred), rows, U, int(seed), int(row_offset), float(left), int(nsamp),
                                              _lib.ptr(t), _lib.current_stream_ptr()), "bnn_sample_instability")
    return t


def summarize_instability(t: torch.Tensor, pred: torch.Tensor, n_trios: int = 1):
    """t [N*n_trios, U], pred [N*n_trios, U, 2] -> [N, 8] (STAT_NAMES)."""
    lib = _lib.load()
    _lib.require_cuda(t, "t")
    t, pred = t.contiguous().float(), pred.contiguous().float()
    rows, U = t.shape
    if rows % n_trios:
        raise ValueError(f"{rows} rows are not a multiple of {n_trios} trios")
    N = rows // n_trios
    stats = torch.empty((N, 8), device=t.device, dtype=torch.float32)
    if N == 0:
        return stats
    with torch.cuda.device(t.device), _lib.nvtx("bnn:K7 summarize_instability"):
        _lib.check(lib.bnn_summarize_instability(_lib.ptr(t), _lib.ptr(pred), N, int(n_trios), U, _lib.ptr(stats),
                                                 _lib.current_stream_ptr()), "bnn_summarize_instability")
    return stats


def posterior_summary(pred: torch.Tensor, n_trios: int = 1, seed: int = 0, row_offset: int = 0):
    """[N*n_trios, U, 2] predictions -> [N, 8] summary (sampling + min over trios + order statistics)."""
    return summarize_instability(sample_instability(pred, seed, row_offset), pred, n_trios)


SCORE_NAMES = ("lpd", "mean_nll")


def score_labels(pred: torch.Tensor, y: torch.Tensor):
    """pred [N, U, 2] (system-major (mu, std)), y [N, 2] labels -> [N, 2] (SCORE_NAMES): per system, the log of the
    ensemble's mean likelihood of the label pair, log((1/U) sum_u exp(-loss_u)), and the mean loss, with loss_u the
    model's own truncated-normal loss (VarModel._lossfnc, ``bnn_nll_fwd_bwd``) of unit u.  Both in nats."""
    if pred.dim() != 3 or pred.shape[2] != 2:
        raise ValueError(f"pred must be [N, U, 2], got {tuple(pred.shape)}")
    N, U = pred.shape[0], pred.shape[1]
    if tuple(y.shape) != (N, 2):
        raise ValueError(f"y must be [{N}, 2] (two labels per system), got {tuple(y.shape)}")
    if U == 0:
        raise ValueError("pred has no units to score")
    lib = _lib.load()
    _lib.require_cuda(pred, "pred")
    pred, y = pred.contiguous().float(), y.contiguous().float()
    score = torch.empty((N, 2), device=pred.device, dtype=torch.float32)
    if N == 0:
        return score
    with torch.cuda.device(pred.device), _lib.nvtx("bnn:K7 score_labels"):
        _lib.check(lib.bnn_score_labels(_lib.ptr(pred), N, U, _lib.dev_ptr(y, pred.device, "y"), _lib.ptr(score),
                                        _lib.current_stream_ptr()), "bnn_score_labels")
    return score


MAX_THRESHOLDS = 64


def survival_thresholds(thresholds) -> np.ndarray:
    """The thresholds of ``survival`` as the kernel compares them: a float32 array of 1 to 64 values, none NaN (+-inf
    allowed).  Raises ValueError otherwise."""
    thr = np.array([float(v) for v in thresholds], np.float32)
    if not 1 <= thr.size <= MAX_THRESHOLDS:
        raise ValueError(f"between 1 and {MAX_THRESHOLDS} thresholds are needed, got {thr.size}")
    if np.isnan(thr).any():
        raise ValueError(f"thresholds must not be NaN, got {thr.tolist()}")
    return thr


def survival(t: torch.Tensor, thresholds, n_trios: int = 1):
    """t [N*n_trios, U] sampled log10 instability times (``sample_instability``), thresholds [J] (log10 orbits, host
    values, rounded to fp32) -> [N, J]: the fraction of the U weight samples whose min over trios exceeds each
    threshold, S_j = #{u : min_r t > thr_j} / U.  S_j is a Monte Carlo estimate of P(T_inst > thr_j) with standard error
    sqrt(S_j (1 - S_j) / U); it counts the same draws as ``summarize_instability``'s percentiles."""
    if t.dim() != 2:
        raise ValueError(f"t must be [N*n_trios, U], got {tuple(t.shape)}")
    if int(n_trios) < 1:
        raise ValueError(f"n_trios must be >= 1, got {n_trios}")
    rows, U = t.shape
    if rows % n_trios:
        raise ValueError(f"{rows} rows are not a multiple of {n_trios} trios")
    if U == 0:
        raise ValueError("t has no units to count")
    thr = survival_thresholds(thresholds)
    lib = _lib.load()
    _lib.require_cuda(t, "t")
    t = t.contiguous().float()
    N = rows // n_trios
    surv = torch.empty((N, thr.size), device=t.device, dtype=torch.float32)
    if N == 0:
        return surv
    h_thr = (ctypes.c_float * thr.size)(*thr.tolist())
    with torch.cuda.device(t.device), _lib.nvtx("bnn:K7 survival_instability"):
        _lib.check(lib.bnn_survival_instability(_lib.ptr(t), N, int(n_trios), U, h_thr, thr.size, _lib.ptr(surv),
                                                _lib.current_stream_ptr()), "bnn_survival_instability")
    return surv


UNCERTAINTY_NAMES = ("mean_mu", "aleatoric", "epistemic", "between_models", "within_models")
MAX_UNCERTAINTY_MODELS = 1024


def uncertainty(pred: torch.Tensor, units_per_model: int):
    """pred [rows, U, 2] (system-major (mu, sigma), unit u = model * units_per_model + sample as
    ``MultiSWAG.sample_thetas`` numbers them) -> [rows, 5] (UNCERTAINTY_NAMES), per row in log10 orbits squared:
    with m_k the mean mu of model k's S = units_per_model samples and mean the mean of the M = U / S model means,
    ``mean_mu`` = mean, ``aleatoric`` = mean sigma^2, ``between_models`` = (1/M) sum_k (m_k - mean)^2,
    ``within_models`` = (1/M) sum_k (1/S) sum_s (mu_{k,s} - m_k)^2 and ``epistemic`` = between + within
    = (1/U) sum_u (mu_u - mean)^2.  Population (ddof = 0) moments, so by the law of total variance the equal-weight
    mixture of the U predicted normals has variance aleatoric + epistemic.  They describe those untruncated normals, not
    the sampled times of ``sample_instability`` (truncated at 4, resampled from the prior above 9, min over trios).
    Accumulated in double, two-pass, rounded once.  A non-finite mu makes every column but ``aleatoric`` NaN; a
    non-finite sigma makes ``aleatoric`` NaN."""
    if pred.dim() != 3 or pred.shape[2] != 2:
        raise ValueError(f"pred must be [rows, U, 2], got {tuple(pred.shape)}")
    rows, U = pred.shape[0], pred.shape[1]
    S = int(units_per_model)
    if U == 0:
        raise ValueError("pred has no units")
    if S < 1 or U % S:
        raise ValueError(f"{U} units are not a positive multiple of units_per_model = {units_per_model}")
    if U // S > MAX_UNCERTAINTY_MODELS:
        raise ValueError(f"{U // S} models: at most {MAX_UNCERTAINTY_MODELS} are supported")
    lib = _lib.load()
    _lib.require_cuda(pred, "pred")
    pred = pred.contiguous().float()
    out = torch.empty((rows, 5), device=pred.device, dtype=torch.float32)
    if rows == 0:
        return out
    with torch.cuda.device(pred.device), _lib.nvtx("bnn:K7 decompose_uncertainty"):
        _lib.check(lib.bnn_decompose_uncertainty(_lib.ptr(pred), rows, U, S, _lib.ptr(out), _lib.current_stream_ptr()),
                   "bnn_decompose_uncertainty")
    return out

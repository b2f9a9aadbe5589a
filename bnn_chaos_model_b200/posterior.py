"""Posterior post-processing on the GPU (SURVEY.md section 8f, rank 1).

Replaces the host-side numpy tail of the reference's evaluation scripts -- ``fast_truncnorm`` (left = 4),
resampling of draws >= 9 from the analytic prior, min over trios, per-system median / percentiles
(figures/main_figures.py:167-277, figures/multiswag_5_planet.py:306-481) -- so that only ``[N, 8]`` leaves the
device instead of the ``[N, U, 2]`` prediction block.  ``survival`` counts the same sampled times against thresholds:
P(T_inst > t) per system.  ``uncertainty`` splits each row's predictive variance into aleatoric, between-model and
within-model parts.

A catalogue of systems with different numbers of planets (P planets: P - 2 adjacent trios) is passed to ``summarize_instability``
and ``survival`` as per-system trio counts instead of one ``n_trios``: system n owns the next counts[n] rows, system-major
as before (``row_offsets``).
"""
from __future__ import annotations

import ctypes
from typing import Optional

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


def is_ragged(n_trios) -> bool:
    """True when ``n_trios`` is per-system trio counts (a sequence, array or tensor with a dimension) rather than one
    count for every system."""
    if isinstance(n_trios, torch.Tensor):
        return n_trios.dim() != 0
    return not isinstance(n_trios, (int, np.integer)) and np.ndim(n_trios) != 0


def row_offsets(counts, rows: Optional[int]) -> np.ndarray:
    """Per-system trio counts c [N] of a catalogue of ``rows`` rows -> row offsets [0, cumsum(c)] (int64 [N + 1]): system
    n owns rows off[n] .. off[n+1] - 1.  Raises ValueError when the counts are not 1-D, are empty, are not integers,
    contain a count below 1, or do not sum to ``rows`` (not checked when ``rows`` is None)."""
    if isinstance(counts, torch.Tensor):
        counts = counts.detach().cpu().numpy()
    c = np.asarray(counts)
    if c.ndim != 1:
        raise ValueError(f"trio counts must be 1-D, got shape {c.shape}")
    if c.size == 0:
        raise ValueError("trio counts are empty: a catalogue needs at least one system")
    if c.dtype == np.bool_ or not np.issubdtype(c.dtype, np.integer):
        raise ValueError(f"trio counts must be integers, got dtype {c.dtype}")
    if (c < 1).any():
        raise ValueError(f"every system needs at least one trio row, got a count of {int(c.min())}")
    off = np.zeros(c.size + 1, np.int64)
    np.cumsum(c, out=off[1:])
    if rows is not None and off[-1] != rows:
        raise ValueError(f"trio counts sum to {int(off[-1])} rows but there are {rows}")
    return off


def device_offsets(off: np.ndarray, device) -> torch.Tensor:
    return torch.from_numpy(np.ascontiguousarray(off, np.int64)).to(device)


def summarize_ragged(t: torch.Tensor, pred: torch.Tensor, d_off: torch.Tensor):
    """``summarize_instability`` of the systems whose row offsets are the device int64 tensor d_off [n + 1], rows
    counted from d_off[0] (``bnn_summarize_instability_ragged``; the offsets are trusted: validate them with
    ``row_offsets``) -> [n, 8]."""
    lib = _lib.load()
    N, U = d_off.shape[0] - 1, t.shape[1]
    stats = torch.empty((N, 8), device=t.device, dtype=torch.float32)
    if N == 0:
        return stats
    with torch.cuda.device(t.device), _lib.nvtx("bnn:K7 summarize_instability"):
        _lib.check(lib.bnn_summarize_instability_ragged(_lib.ptr(t), _lib.ptr(pred), N,
                                                        _lib.dev_ptr(d_off, t.device, "row offsets", torch.int64), U,
                                                        _lib.ptr(stats), _lib.current_stream_ptr()),
                   "bnn_summarize_instability_ragged")
    return stats


def summarize_instability(t: torch.Tensor, pred: torch.Tensor, n_trios=1):
    """t [N*n_trios, U], pred [N*n_trios, U, 2] -> [N, 8] (STAT_NAMES).  ``n_trios`` may also be per-system trio counts
    [N] (1-D integers >= 1 summing to the rows of t; ``row_offsets``)."""
    if is_ragged(n_trios):
        off = row_offsets(n_trios, t.shape[0])
        _lib.require_cuda(t, "t")
        t, pred = t.contiguous().float(), pred.contiguous().float()
        return summarize_ragged(t, pred, device_offsets(off, t.device))
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


def survival_ragged(t: torch.Tensor, thr: np.ndarray, d_off: torch.Tensor):
    """``survival`` of the systems whose row offsets are the device int64 tensor d_off [n + 1], rows counted from
    d_off[0] (``bnn_survival_instability_ragged``; thr as ``survival_thresholds`` returns it, the offsets trusted) ->
    [n, J]."""
    lib = _lib.load()
    N, U = d_off.shape[0] - 1, t.shape[1]
    surv = torch.empty((N, thr.size), device=t.device, dtype=torch.float32)
    if N == 0:
        return surv
    h_thr = (ctypes.c_float * thr.size)(*thr.tolist())
    with torch.cuda.device(t.device), _lib.nvtx("bnn:K7 survival_instability"):
        _lib.check(lib.bnn_survival_instability_ragged(_lib.ptr(t), N,
                                                       _lib.dev_ptr(d_off, t.device, "row offsets", torch.int64), U, h_thr,
                                                       thr.size, _lib.ptr(surv), _lib.current_stream_ptr()),
                   "bnn_survival_instability_ragged")
    return surv


def survival(t: torch.Tensor, thresholds, n_trios=1):
    """t [N*n_trios, U] sampled log10 instability times (``sample_instability``), thresholds [J] (log10 orbits, host
    values, rounded to fp32) -> [N, J]: the fraction of the U weight samples whose min over trios exceeds each
    threshold, S_j = #{u : min_r t > thr_j} / U.  S_j is a Monte Carlo estimate of P(T_inst > thr_j) with standard error
    sqrt(S_j (1 - S_j) / U); it counts the same draws as ``summarize_instability``'s percentiles.  ``n_trios`` may also
    be per-system trio counts [N] (``row_offsets``)."""
    if t.dim() != 2:
        raise ValueError(f"t must be [N*n_trios, U], got {tuple(t.shape)}")
    if is_ragged(n_trios):
        off = row_offsets(n_trios, t.shape[0])
        if t.shape[1] == 0:
            raise ValueError("t has no units to count")
        thr = survival_thresholds(thresholds)
        _lib.require_cuda(t, "t")
        t = t.contiguous().float()
        return survival_ragged(t, thr, device_offsets(off, t.device))
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

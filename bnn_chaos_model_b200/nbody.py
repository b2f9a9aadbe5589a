"""Predict from initial orbits: the short N-body integration on the device (K8, ``bnn_integrate_orbits``).

A user of the model has orbits and masses, not time series.  ``integrate_orbits`` integrates each system for
``n_orbits`` inner orbits with a WHFast-style Wisdom-Holman kernel in fp64 (one system per thread) and returns the raw
``tseries`` / ``masses`` rows that ``inputs.data_setup_kernel`` packs, one row per adjacent trio, plus the time at which
a system went unstable during the integration.  Only the columns the shipped v50 ensembles read are computed: columns
1-7 (e+-, MMR strength, MEGNO) are 0.  Conventions: csrc/nbody.cu and DESIGN.md, section K8.

Each planet is 7 numbers (m / M_star, a, e, inc, Omega, varpi, lambda), Jacobi elements with G = M_star = 1, planets
ordered from the inside out.
"""
from __future__ import annotations

import math

import numpy as np
import torch

from . import _lib

N_OUT, N_COLS = 100, 26
MIN_PLANETS, MAX_PLANETS = 3, 8
LIVE_COLUMNS_NOT_COMPUTED = tuple(range(1, 8))   # e+- near/far, MMR strength near/far, MEGNO
PER_ROW_KEYS = ("uncertainty", "trio_first", "trio_summary", "attribution", "attribution_mu")


def planet_counts(n_planets, rows: int) -> np.ndarray:
    """Per-system planet counts int64 [N] from an int (every system has that many planets) or counts [N].  Raises
    ValueError when a count is outside 3..8 or the counts do not add up to the element rows."""
    if isinstance(n_planets, (int, np.integer)):
        P = int(n_planets)
        if not MIN_PLANETS <= P <= MAX_PLANETS:
            raise ValueError(f"n_planets = {P} must be in {MIN_PLANETS}..{MAX_PLANETS}")
        if rows % P:
            raise ValueError(f"{rows} planet rows are not a whole number of {P}-planet systems")
        counts = np.full(rows // P, P, dtype=np.int64)
    else:
        c = np.asarray(n_planets.detach().cpu() if isinstance(n_planets, torch.Tensor) else n_planets)
        if c.ndim != 1 or c.size == 0 or not np.issubdtype(c.dtype, np.integer):
            raise ValueError(f"n_planets must be an int or a 1-D integer array of per-system counts, got {c.dtype} "
                             f"{c.shape}")
        if c.min() < MIN_PLANETS or c.max() > MAX_PLANETS:
            raise ValueError(f"planet counts must be in {MIN_PLANETS}..{MAX_PLANETS}, got {int(c.min())}..{int(c.max())}")
        counts = c.astype(np.int64)
    if counts.size == 0 or int(counts.sum()) != rows:
        raise ValueError(f"the planet counts add up to {int(counts.sum())} planets but the elements have {rows} rows")
    return counts


def check_elements(el: np.ndarray, counts: np.ndarray) -> None:
    """ValueError unless every value is finite, m >= 0, a > 0, 0 <= e < 1 and a increases within each system."""
    bad = lambda mask: int(np.flatnonzero(mask)[0])
    if not np.isfinite(el).all():
        raise ValueError(f"orbit row {bad(~np.isfinite(el).all(1))} has a non-finite value")
    m, a, e = el[:, 0], el[:, 1], el[:, 2]
    if (m < 0).any():
        raise ValueError(f"orbit row {bad(m < 0)} has a negative mass {m[m < 0][0]}")
    if (a <= 0).any():
        raise ValueError(f"orbit row {bad(a <= 0)} has a <= 0 ({a[a <= 0][0]})")
    if ((e < 0) | (e >= 1)).any():
        raise ValueError(f"orbit row {bad((e < 0) | (e >= 1))} has e outside [0, 1)")
    first = np.zeros(el.shape[0], bool)
    first[np.concatenate([[0], np.cumsum(counts)[:-1]])] = True
    step = np.concatenate([[np.inf], np.diff(a)])
    if ((step <= 0) & ~first).any():
        raise ValueError(f"orbit row {bad((step <= 0) & ~first)}: semi-major axes must increase within a system")


def check_run(n_orbits: float, dt_frac: float) -> None:
    if not (math.isfinite(n_orbits) and n_orbits > 0 and math.isfinite(dt_frac) and dt_frac > 0):
        raise ValueError(f"n_orbits and dt_frac must be finite and > 0, got {n_orbits}, {dt_frac}")
    if 990.0 * n_orbits / 999.0 / dt_frac > 2.0 ** 31:
        raise ValueError(f"n_orbits / dt_frac = {n_orbits / dt_frac:g} needs more than 2^31 steps")


def integrate_orbits(elements, n_planets, n_orbits: float = 1e4, dt_frac: float = 0.05, device=None):
    """elements [sum P, 7] (or [N, P, 7] with an int ``n_planets``) -> (tseries [R, 100, 26], masses [R, 3],
    log10_t_unstable [N]), float64 CUDA tensors, R = sum (P - 2) trio rows, system-major.

    ``n_planets``: an int, or per-system counts [N] for a catalogue of mixed planet counts; such a catalogue is
    bucketed by planet count on the host, one launch per count, and the rows are scattered back into catalogue order.
    A system's results do not depend on the other systems in the call.  Raises ValueError, before any device work, on
    counts outside 3..8, counts that do not add up to the rows, a <= 0, e outside [0, 1), a not increasing within a
    system, m < 0, non-finite values, or n_orbits / dt_frac that are not finite and > 0."""
    src = elements.detach() if isinstance(elements, torch.Tensor) else None
    el = np.ascontiguousarray((src.cpu().numpy() if src is not None else np.asarray(elements)), dtype=np.float64)
    if el.ndim == 3 and el.shape[2] == 7:
        el = el.reshape(-1, 7)
    if el.ndim != 2 or el.shape[1] != 7 or el.shape[0] == 0:
        raise ValueError(f"elements must be [planets, 7] or [N, P, 7], got {tuple(el.shape)}")
    counts = planet_counts(n_planets, el.shape[0])
    check_elements(el, counts)
    check_run(float(n_orbits), float(dt_frac))
    lib = _lib.load()
    dev = torch.device(device) if device is not None else (
        src.device if src is not None and src.is_cuda else torch.device("cuda", torch.cuda.current_device()))
    N = counts.size
    R = int((counts - 2).sum())
    ts = torch.empty((R, N_OUT, N_COLS), dtype=torch.float64, device=dev)
    ms = torch.empty((R, 3), dtype=torch.float64, device=dev)
    lt = torch.empty(N, dtype=torch.float64, device=dev)
    planet_off = np.concatenate([[0], np.cumsum(counts)])
    row_off = np.concatenate([[0], np.cumsum(counts - 2)])
    uniform = bool((counts == counts[0]).all())
    with torch.cuda.device(dev), _lib.nvtx("bnn:K8 integrate_orbits"):
        stream = _lib.current_stream_ptr()
        for P in np.unique(counts):
            P = int(P)
            systems = np.flatnonzero(counts == P)
            if uniform:
                d_el, d_ts, d_ms, d_lt = torch.from_numpy(el).to(dev), ts, ms, lt
            else:
                planets = (planet_off[systems][:, None] + np.arange(P)).reshape(-1)
                d_el = torch.from_numpy(np.ascontiguousarray(el[planets])).to(dev)
                n = systems.size
                d_ts = torch.empty((n * (P - 2), N_OUT, N_COLS), dtype=torch.float64, device=dev)
                d_ms = torch.empty((n * (P - 2), 3), dtype=torch.float64, device=dev)
                d_lt = torch.empty(n, dtype=torch.float64, device=dev)
            _lib.check(lib.bnn_integrate_orbits(d_el.data_ptr(), systems.size, P, float(n_orbits), float(dt_frac),
                                                d_ts.data_ptr(), d_ms.data_ptr(), d_lt.data_ptr(), stream),
                       "bnn_integrate_orbits")
            if not uniform:
                rows = torch.from_numpy((row_off[systems][:, None] + np.arange(P - 2)).reshape(-1)).to(dev)
                ts.index_copy_(0, rows, d_ts)
                ms.index_copy_(0, rows, d_ms)
                lt.index_copy_(0, torch.from_numpy(systems).to(dev), d_lt)
    return ts, ms, lt


def check_zero_mask(models) -> None:
    """ValueError unless every model zeroes the input columns the integration does not compute (1-7)."""
    for k, m in enumerate(models):
        missing = sorted(set(LIVE_COLUMNS_NOT_COMPUTED) - set(m.zero_columns()))
        if missing:
            raise ValueError(f"model {k} reads input columns {missing} (e+-, MMR strength or MEGNO), which the orbit "
                             "integration does not compute: an orbit catalogue needs an ensemble whose flags zero "
                             "columns 1-7 (include_mmr = include_eplusminus = False, fix_megno2)")


def override_unstable(arrays: dict, log10_t_unstable, n_trios) -> dict:
    """Apply the known instability times of systems that went unstable during the integration to the posterior outputs
    (a copy of ``arrays``, the per_system.npz entries of ``predict``): for each system with a finite
    ``log10_t_unstable`` t, summary columns 0-5 = t and 6-7 = NaN; survival[:, j] = 1.0 if t > thresholds[j] else
    0.0; its trio rows of ``uncertainty``, ``trio_first``, ``trio_summary``, ``attribution`` and ``attribution_mu`` =
    NaN.  Other systems and other keys are unchanged."""
    from .posterior import row_offsets

    lt = np.asarray(log10_t_unstable, dtype=np.float64)
    off = row_offsets(np.asarray(n_trios), None)
    N, R = off.size - 1, int(off[-1])
    if lt.shape != (N,):
        raise ValueError(f"log10_t_unstable must be [{N}] (one per system), got {lt.shape}")
    if "summary" not in arrays or arrays["summary"].shape != (N, 8):
        raise ValueError(f"arrays need summary [{N}, 8]")
    if "survival" in arrays and "thresholds" not in arrays:
        raise ValueError("survival needs its thresholds")
    out = dict(arrays)
    hit = np.isfinite(lt)
    s = np.array(arrays["summary"], copy=True)
    s[hit, :6] = lt[hit, None].astype(s.dtype)
    s[hit, 6:] = np.nan
    out["summary"] = s
    if "survival" in arrays:
        sv = np.array(arrays["survival"], copy=True)
        thr = np.asarray(arrays["thresholds"], dtype=np.float64)
        if sv.shape != (N, thr.size):
            raise ValueError(f"survival must be [{N}, {thr.size}], got {sv.shape}")
        sv[hit] = (lt[hit, None] > thr[None, :]).astype(sv.dtype)
        out["survival"] = sv
    rows = np.repeat(hit, np.diff(off))
    for k in PER_ROW_KEYS:
        if k in arrays:
            a = np.array(arrays[k], copy=True)
            if a.shape[0] != R:
                raise ValueError(f"{k} must have one entry per trio row ({R}), got {a.shape}")
            a[rows] = np.nan
            out[k] = a
    return out

"""CPU: the survival probability's oracle, the argument checks of posterior.survival / MultiSWAG.posterior_survival
(raised before any device work) and of the C entry bnn_survival_instability (returned before the device is queried), and
the evaluate CLI's --survival flag and Brier score."""
import ctypes

import numpy as np
import pytest
import torch

from bnn_chaos_model_b200 import _lib, evaluate
from bnn_chaos_model_b200._lib import BnnChaosError
from bnn_chaos_model_b200.multiswag import MultiSWAG
from bnn_chaos_model_b200.posterior import MAX_THRESHOLDS, survival, survival_thresholds
from oracle.survival import survival_fraction

INF, NAN = np.inf, np.nan


def test_oracle_counts_strictly_above_each_threshold():
    t = np.array([[4.5, 9.0, 9.0, 12.0, -INF, INF, NAN, 6.0]], np.float32)
    got = survival_fraction(t, [-INF, 4.5, 9.0, 11.0, INF, 6.0])
    # tmin = t (one trio); NaN is +inf like the summary's fmin from +inf
    assert got.dtype == np.float32 and got.shape == (1, 6)
    assert got.tolist() == [[7 / 8, 6 / 8, 3 / 8, 3 / 8, 0.0, 5 / 8]]


def test_oracle_takes_the_min_over_trios_with_fmin_from_inf():
    # rows = system * 3 + trio.  System 0, units 0..2 over its trios: (5, NaN, 7) -> 5; (NaN, NaN, NaN) -> +inf;
    # (10, 3, NaN) -> 3.  System 1: every draw NaN.
    t = np.array([[5.0, NAN, 10.0], [NAN, NAN, 3.0], [7.0, NAN, NAN],
                  [NAN, NAN, NAN], [NAN, NAN, NAN], [NAN, NAN, NAN]], np.float32)
    got = survival_fraction(t, [4.0, 9.0, INF], n_trios=3)
    tmin0 = np.array([5.0, INF, 3.0])
    assert got[0].tolist() == [np.float32(np.mean(tmin0 > 4.0)), np.float32(np.mean(tmin0 > 9.0)), 0.0]
    assert got[1].tolist() == [1.0, 1.0, 0.0]   # every unit all-NaN: +inf, above any finite threshold


def test_oracle_rounds_the_exact_fraction_once():
    rng = np.random.default_rng(0)
    U = 60000
    t = rng.uniform(4, 12, (3, U)).astype(np.float32)
    thr = np.array([5.0, 7.5, 9.0], np.float32)
    got = survival_fraction(t, thr)
    count = (t[:, :, None] > thr).sum(1)
    assert np.array_equal(got, (count / U).astype(np.float32))
    assert np.array_equal(got, survival_fraction(t[:, rng.permutation(U)], thr))   # order of the draws is irrelevant


def test_survival_thresholds_validation():
    assert survival_thresholds([9]).tolist() == [9.0] and survival_thresholds((-INF, INF)).tolist() == [-INF, INF]
    assert survival_thresholds(np.arange(64.0)).dtype == np.float32 and MAX_THRESHOLDS == 64
    for bad in ([], np.arange(65.0), [4.0, NAN]):
        with pytest.raises(ValueError):
            survival_thresholds(bad)


def test_survival_argument_errors():
    t = torch.zeros((6, 5))
    for tt, thr, R in ((torch.zeros(6), [9.0], 1), (torch.zeros((6, 5, 1)), [9.0], 1), (t, [9.0], 4), (t, [9.0], 0),
                       (torch.zeros((6, 0)), [9.0], 1), (t, [], 1), (t, list(range(65)), 1), (t, [NAN], 1)):
        with pytest.raises(ValueError):
            survival(tt, thr, R)
    with pytest.raises(BnnChaosError):   # CPU tensors: no fallback
        survival(t, [9.0], 3)


def bare_ensemble():
    """A MultiSWAG without any state: any device work in the method under test would fail with AttributeError."""
    return object.__new__(MultiSWAG)


@pytest.mark.parametrize("x,thr,S,R,match", [
    (torch.zeros((6, 100)), [9.0], 3, 1, "x must be"),
    (torch.zeros((7, 100, 41)), [9.0], 3, 3, "not a multiple"),
    (torch.zeros((6, 100, 41)), [9.0], 3, 0, "not a multiple"),
    (torch.zeros((6, 100, 41)), [9.0], 0, 3, "samples_per_model"),
    (torch.zeros((6, 100, 41)), [], 3, 1, "thresholds"),
    (torch.zeros((6, 100, 41)), list(range(65)), 3, 1, "thresholds"),
    (torch.zeros((6, 100, 41)), [9.0, NAN], 3, 1, "NaN"),
])
def test_posterior_survival_argument_errors_before_device_work(x, thr, S, R, match):
    with pytest.raises(ValueError, match=match):
        bare_ensemble().posterior_survival(x, thr, S, n_trios=R)
    with pytest.raises(ValueError, match=match):
        bare_ensemble().posterior_survival_sharded(x, thr, 2, S, n_trios=R)


def test_posterior_survival_rejects_cpu_tensors():
    with pytest.raises(BnnChaosError):
        bare_ensemble().posterior_survival(torch.zeros((6, 100, 41)), [9.0], 3, n_trios=3)


def test_survival_entry_argument_errors():
    """BNN_E_ARG / BNN_E_ALIGN come back before the device is queried; the fake device addresses are never
    dereferenced."""
    lib = _lib.load()
    tp, sp = 1 << 20, 2 << 20
    thr = (ctypes.c_float * 3)(4.0, 9.0, NAN)
    for args in ((None, 4, 1, 10, thr, 2, sp), (tp, 4, 1, 10, None, 2, sp), (tp, 4, 1, 10, thr, 2, None),
                 (tp, 0, 1, 10, thr, 2, sp), (tp, -1, 1, 10, thr, 2, sp), (tp, 4, 1, 0, thr, 2, sp),
                 (tp, 4, 1, -3, thr, 2, sp), (tp, 4, 0, 10, thr, 2, sp), (tp, 4, -2, 10, thr, 2, sp),
                 (tp, 4, 1, 10, thr, 0, sp), (tp, 4, 1, 10, thr, -1, sp), (tp, 4, 1, 10, thr, 65, sp),
                 (tp, 1 << 31, 1, 10, thr, 2, sp), (tp, 4, 1, 1 << 32, thr, 2, sp),
                 (tp, 4, 1, 10, thr, 3, sp)):   # the third threshold is NaN
        assert lib.bnn_survival_instability(*args, None) == -1, args   # BNN_E_ARG
        assert lib.bnn_last_error_string().startswith(b"bnn_survival_instability")
    assert b"NaN" in lib.bnn_last_error_string()
    for args in ((tp + 2, 4, 1, 10, thr, 2, sp), (tp, 4, 1, 10, thr, 2, sp + 1)):
        assert lib.bnn_survival_instability(*args, None) == -4, args   # BNN_E_ALIGN
        assert b"aligned" in lib.bnn_last_error_string()


def test_evaluate_cli_survival_flag():
    ap = evaluate.build_parser()
    assert ap.parse_args(["--models", "m.pkl", "--out", "o"]).survival is None
    a = ap.parse_args(["--models", "m.pkl", "--out", "o", "--survival", "6", "9"])
    assert a.survival == [6.0, 9.0]
    assert ap.parse_args(["--models", "m.pkl", "--survival", "4", "9.5", "inf", "--out", "o"]).survival == [4.0, 9.5, INF]
    for bad in (["--survival"], ["--survival", "x"]):
        with pytest.raises(SystemExit):
            ap.parse_args(["--models", "m.pkl", "--out", "o"] + bad)
    for bad in (["nan"], [str(v) for v in range(65)]):   # rejected before any device work
        with pytest.raises(ValueError):
            evaluate.main(["--models", "m.pkl", "--out", "o", "--survival"] + bad)


def test_brier_stable():
    s9 = np.array([0.25, 1.0, 0.0, 0.5], np.float32)
    y = np.array([[9.0, 5.0], [NAN, 12.0], [4.5, NAN], [NAN, NAN]], np.float32)
    brier, n_stable = evaluate.brier_stable(s9, y)
    assert n_stable == 2
    assert brier == pytest.approx(((0.25 - 1) ** 2 + 0.25 ** 2 + 0.0 + 0.0) / 4, rel=1e-15)
    assert evaluate.brier_stable(s9[3:], y[3:]) == (None, 0)

"""CPU: the variance decomposition's oracle (identity, exact zeros, NaN rules), the argument checks of
posterior.uncertainty / MultiSWAG.posterior_uncertainty (raised before any device work) and of the C entry
bnn_decompose_uncertainty (returned before the device is queried), and the evaluate CLI's --uncertainty flag."""
import numpy as np
import pytest
import torch

from bnn_chaos_model_b200 import _lib, evaluate
from bnn_chaos_model_b200._lib import BnnChaosError
from bnn_chaos_model_b200.multiswag import MultiSWAG
from bnn_chaos_model_b200.posterior import MAX_UNCERTAINTY_MODELS, UNCERTAINTY_NAMES, uncertainty
from oracle.uncertainty import epistemic_direct, variance_decomposition

INF, NAN = np.inf, np.nan


def random_pred(rows, M, S, seed):
    rng = np.random.default_rng(seed)
    return np.stack([rng.uniform(4, 12, (rows, M * S)), rng.uniform(0.5, 6, (rows, M * S))], -1).astype(np.float32)


def test_oracle_by_hand():
    # two models of two samples: mu (4, 6 | 8, 10) -> m = (5, 9), mean 7; between = 4, within = 1
    pred = np.array([[[4.0, 1.0], [6.0, 2.0], [8.0, 3.0], [10.0, 4.0]]], np.float32)
    got = variance_decomposition(pred, 2)
    assert got.dtype == np.float32 and got.shape == (1, 5)
    assert got.tolist() == [[7.0, (1 + 4 + 9 + 16) / 4, 5.0, 4.0, 1.0]]
    assert UNCERTAINTY_NAMES == ("mean_mu", "aleatoric", "epistemic", "between_models", "within_models")


@pytest.mark.parametrize("M,S", [(1, 7), (3, 1), (5, 7), (30, 100)])
def test_oracle_law_of_total_variance(M, S):
    pred = random_pred(6, M, S, M * S)
    got = variance_decomposition(pred, S)
    direct = epistemic_direct(pred)
    assert np.allclose(direct, np.var(pred[:, :, 0].astype(np.float64), 1), rtol=1e-12, atol=0)   # ddof = 0
    assert (np.abs(got[:, 2] - direct) <= np.spacing(got[:, 2])).all()
    assert (np.abs(got[:, 2] - (got[:, 3].astype(np.float64) + got[:, 4])) <= 2 * np.spacing(got[:, 2])).all()
    assert np.allclose(got[:, 1], (pred[:, :, 1].astype(np.float64) ** 2).mean(1), rtol=1e-7, atol=0)


def test_oracle_exact_zeros():
    pred = random_pred(3, 4, 5, 1)
    assert (variance_decomposition(pred[:, :5], 5)[:, 3] == 0).all()    # M = 1
    assert (variance_decomposition(pred, 1)[:, 4] == 0).all()           # S = 1
    pred[1, :, 0] = 7.3
    got = variance_decomposition(pred, 5)[1]
    assert got[0] == np.float32(7.3) and (got[2:] == 0).all() and got[1] > 0


def test_oracle_nan_rules():
    pred = random_pred(4, 3, 5, 2)
    pred[0, 3, 0] = NAN
    pred[1, 7, 1] = INF
    pred[2, 0, 0] = INF
    pred[2, 1, 1] = NAN
    got = variance_decomposition(pred, 5)
    ref = variance_decomposition(pred[3:], 5)
    assert np.isnan(got[0, [0, 2, 3, 4]]).all() and np.isfinite(got[0, 1])
    assert np.isnan(got[1, 1]) and np.isfinite(got[1, [0, 2, 3, 4]]).all()
    assert np.isnan(got[2]).all()
    assert np.array_equal(got[3], ref[0])


def test_uncertainty_argument_errors():
    p = torch.zeros((4, 12, 2))
    for pp, S in ((torch.zeros((4, 12)), 1), (torch.zeros((4, 12, 3)), 1), (torch.zeros((4, 0, 2)), 1), (p, 0), (p, -3),
                  (p, 5), (p, 24), (torch.zeros((2, MAX_UNCERTAINTY_MODELS + 1, 2)), 1)):
        with pytest.raises(ValueError):
            uncertainty(pp, S)
    assert MAX_UNCERTAINTY_MODELS == 1024
    with pytest.raises(BnnChaosError):   # CPU tensors: no fallback
        uncertainty(torch.zeros((2, MAX_UNCERTAINTY_MODELS * 2, 2)), 2)


def bare_ensemble():
    """A MultiSWAG without any state: any device work in the method under test would fail with AttributeError."""
    return object.__new__(MultiSWAG)


@pytest.mark.parametrize("x,S,R,match", [
    (torch.zeros((6, 100)), 3, 1, "x must be"),
    (torch.zeros((7, 100, 41)), 3, 3, "not a multiple"),
    (torch.zeros((6, 100, 41)), 3, 0, "not a multiple"),
    (torch.zeros((6, 100, 41)), 0, 3, "samples_per_model"),
])
def test_posterior_uncertainty_argument_errors_before_device_work(x, S, R, match):
    with pytest.raises(ValueError, match=match):
        bare_ensemble().posterior_uncertainty(x, S, n_trios=R)
    with pytest.raises(ValueError, match=match):
        bare_ensemble().posterior_uncertainty_sharded(x, 2, S, n_trios=R)


def test_posterior_uncertainty_rejects_cpu_tensors():
    with pytest.raises(BnnChaosError):
        bare_ensemble().posterior_uncertainty(torch.zeros((6, 100, 41)), 3, n_trios=3)


def test_uncertainty_entry_argument_errors():
    """BNN_E_ARG / BNN_E_ALIGN come back before the device is queried; the fake device addresses are never
    dereferenced."""
    lib = _lib.load()
    pp, op = 1 << 20, 2 << 20
    for args in ((None, 4, 12, 3, op), (pp, 4, 12, 3, None), (pp, 0, 12, 3, op), (pp, -1, 12, 3, op),
                 (pp, 1 << 31, 12, 3, op), (pp, 4, 0, 1, op), (pp, 4, -6, 3, op), (pp, 4, 1 << 32, 1 << 31, op),
                 (pp, 4, 12, 0, op), (pp, 4, 12, -3, op), (pp, 4, 12, 5, op), (pp, 4, 12, 24, op),
                 (pp, 4, 1025, 1, op), (pp, 4, 1025 * 7, 7, op)):
        assert lib.bnn_decompose_uncertainty(*args, None) == -1, args   # BNN_E_ARG
        assert lib.bnn_last_error_string().startswith(b"bnn_decompose_uncertainty"), args
    assert b"1025 models" in lib.bnn_last_error_string()
    for args in ((pp + 4, 4, 12, 3, op), (pp, 4, 12, 3, op + 2), (pp + 1, 4, 12, 3, op)):
        assert lib.bnn_decompose_uncertainty(*args, None) == -4, args   # BNN_E_ALIGN
        assert lib.bnn_last_error_string().startswith(b"bnn_decompose_uncertainty")
        assert b"aligned" in lib.bnn_last_error_string()


def test_evaluate_cli_uncertainty_flag():
    ap = evaluate.build_parser()
    assert ap.parse_args(["--models", "m.pkl", "--out", "o"]).uncertainty is False
    assert ap.parse_args(["--models", "m.pkl", "--out", "o", "--uncertainty"]).uncertainty is True
    a = ap.parse_args(["--models", "m.pkl", "--uncertainty", "--survival", "6", "9", "--out", "o"])
    assert a.uncertainty is True and a.survival == [6.0, 9.0]
    with pytest.raises(SystemExit):
        ap.parse_args(["--models", "m.pkl", "--out", "o", "--uncertainty", "1"])

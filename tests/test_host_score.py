"""CPU: the held-out score's oracle, the argument checks of score_labels / MultiSWAG.evaluate (raised before any device
work) and of the C entry bnn_score_labels (returned before the device is queried), and the evaluate CLI's parser."""
import numpy as np
import pytest
import torch
from scipy.special import logsumexp

from bnn_chaos_model_b200 import _lib, evaluate
from bnn_chaos_model_b200._lib import BnnChaosError
from bnn_chaos_model_b200.multiswag import MultiSWAG
from bnn_chaos_model_b200.posterior import SCORE_NAMES, score_labels
from oracle import restatement as R
from oracle.score import predictive_score


def random_block(N, U, seed):
    rng = np.random.default_rng(seed)
    pred = np.stack([rng.uniform(4, 12, (N, U)), rng.uniform(0.1, 6, (N, U))], -1).astype(np.float32)
    y = rng.uniform(4, 14, (N, 2)).astype(np.float32)
    y[0] = (5.0, 9.0)   # exactly at the censoring threshold
    return pred, y


def test_oracle_single_unit_is_the_loss():
    pred, y = random_block(50, 1, 1)
    loss = R.lossfnc_per_system(torch.from_numpy(pred[:, 0]), torch.from_numpy(y)).double().numpy()
    got = predictive_score(pred, y)
    assert got.dtype == np.float64 and got.shape == (50, 2)
    assert np.array_equal(got[:, 0], -loss) and np.array_equal(got[:, 1], loss)


def test_oracle_is_a_log_mean_exp_invariant_to_unit_order():
    pred, y = random_block(20, 300, 2)
    pred[3, :, 0] = np.nan       # every unit of a row on the -100 guard, both labels
    pred[4, 7] = np.nan
    y[5] = np.nan
    got = predictive_score(pred, y)
    assert np.isfinite(got).all()
    loss = R.lossfnc_per_system(torch.from_numpy(pred.reshape(-1, 2)), torch.from_numpy(np.repeat(y, 300, 0)))
    loss = loss.double().numpy().reshape(20, 300)
    np.testing.assert_allclose(got[:, 0], logsumexp(-loss, axis=1) - np.log(300), rtol=1e-13, atol=1e-13)
    np.testing.assert_allclose(got[:, 1], loss.mean(1), rtol=1e-13)
    assert got[3, 0] == -200.0 and got[3, 1] == 200.0
    assert got[5, 0] == -200.0 and got[5, 1] == 200.0
    perm = np.random.default_rng(3).permutation(300)
    np.testing.assert_allclose(predictive_score(pred[:, perm], y), got, rtol=1e-13, atol=1e-13)


def test_score_labels_argument_errors():
    assert SCORE_NAMES == ("lpd", "mean_nll")
    pred, y = torch.zeros((4, 3, 2)), torch.zeros((4, 2))
    for p, yy in ((torch.zeros((4, 3)), y), (torch.zeros((4, 3, 3)), y), (pred, torch.zeros((3, 2))),
                  (pred, torch.zeros((4, 1))), (torch.zeros((4, 0, 2)), y)):
        with pytest.raises(ValueError):
            score_labels(p, yy)
    with pytest.raises(BnnChaosError):   # CPU tensors: no fallback
        score_labels(pred, y)


def bare_ensemble():
    """A MultiSWAG without any state: any device work in the method under test would fail with AttributeError."""
    return object.__new__(MultiSWAG)


@pytest.mark.parametrize("x,y,S,match", [
    (torch.zeros((5, 100)), torch.zeros((5, 2)), 3, "x must be"),
    (torch.zeros((5, 100, 41)), torch.zeros((5,)), 3, "y must be"),
    (torch.zeros((5, 100, 41)), torch.zeros((5, 3)), 3, "y must be"),
    (torch.zeros((5, 100, 41)), torch.zeros((4, 2)), 3, "4 rows"),
    (torch.zeros((5, 100, 41)), torch.zeros((5, 2)), 0, "samples_per_model"),
])
def test_evaluate_argument_errors_before_device_work(x, y, S, match):
    with pytest.raises(ValueError, match=match):
        bare_ensemble().evaluate(x, y, S)
    with pytest.raises(ValueError, match=match):
        bare_ensemble().evaluate_sharded(x, y, 5, S)


def test_evaluate_rejects_cpu_tensors():
    with pytest.raises(BnnChaosError):
        bare_ensemble().evaluate(torch.zeros((5, 100, 41)), torch.zeros((5, 2)), 3)


def test_score_entry_argument_errors():
    """BNN_E_ARG / BNN_E_ALIGN come back before the device is queried; the fake addresses are never dereferenced."""
    lib = _lib.load()
    p, yv, s = 1 << 20, 2 << 20, 3 << 20
    for args in ((None, 4, 3, yv, s), (p, 4, 3, None, s), (p, 4, 3, yv, None), (p, 0, 3, yv, s), (p, -1, 3, yv, s),
                 (p, 4, 0, yv, s), (p, 4, -5, yv, s), (p, 1 << 31, 3, yv, s), (p, 4, 1 << 32, yv, s)):
        assert lib.bnn_score_labels(*args, None) == -1, args   # BNN_E_ARG
        assert lib.bnn_last_error_string().startswith(b"bnn_score_labels")
    for args in ((p + 4, 4, 3, yv, s), (p, 4, 3, yv + 4, s), (p, 4, 3, yv, s + 2)):
        assert lib.bnn_score_labels(*args, None) == -4, args   # BNN_E_ALIGN
        assert b"aligned" in lib.bnn_last_error_string()


def test_evaluate_cli_parser():
    ap = evaluate.build_parser()
    a = ap.parse_args(["--models", "a_output.pkl", "b_output.pkl", "--out", "o"])
    assert a.models == ["a_output.pkl", "b_output.pkl"] and a.out == "o"
    assert (a.data, a.synthetic, a.samples, a.seed, a.scale) == (None, 1000, 100, 0, 0.5)
    a = ap.parse_args(["--models", "m.pkl", "--data", "d.npz", "--samples", "7", "--seed", "4", "--scale", "0.25",
                       "--out", "o"])
    assert (a.data, a.samples, a.seed, a.scale) == ("d.npz", 7, 4, 0.25)
    for bad in ([], ["--out", "o"], ["--models", "m.pkl"], ["--models", "m.pkl", "--out", "o", "--samples", "x"]):
        with pytest.raises(SystemExit):
            ap.parse_args(bad)

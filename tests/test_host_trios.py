"""CPU: which trio goes unstable first -- the first-trio oracle's rules on hand-built cases, the Python argument checks
(before any device work), the C entries' argument and alignment errors (returned before the device is queried), and
the predict CLI's --trios flag."""
import numpy as np
import pytest
import torch

from bnn_chaos_model_b200 import _lib, predict
from bnn_chaos_model_b200.multiswag import MultiSWAG
from bnn_chaos_model_b200.posterior import MAX_TRIOS_PER_SYSTEM, check_trio_counts, first_trio
from oracle.trios import catalogue_first_trio

INF, NAN = np.inf, np.nan


def test_oracle_rules():
    # counts [1, 3, 2], units in columns.  System 0: one trio wins every unit.  System 1: unit 0 a clear min (row 2),
    # unit 1 a tie between rows 1 and 2 (the earlier wins), unit 2 NaN in row 1 is ignored, unit 3 all NaN (no
    # winner), unit 4 all +inf or NaN (the first +inf row wins), unit 5 +inf loses to a finite draw.  System 2: unit 0
    # tie -> row 0, unit 1 NaN / 6 -> row 1, unit 2 all NaN, unit 3 +inf / +inf -> row 0, units 4, 5 plain.
    t = np.array([[5.0, 6.0, 7.0, 8.0, 9.0, 4.0],
                  [6.0, 5.0, NAN, NAN, NAN, INF],
                  [7.0, 5.0, 4.5, NAN, INF, 7.5],
                  [4.0, 6.0, 5.0, NAN, INF, INF],
                  [5.0, NAN, NAN, INF, 4.0, 9.0],
                  [5.0, 6.0, NAN, INF, 5.0, 8.0]], np.float32)
    got = catalogue_first_trio(t, [1, 3, 2])
    assert got.dtype == np.float32 and got.shape == (6,)
    U = 6
    assert (got * U).round().astype(int).tolist() == [6, 1, 3, 1, 3, 2]
    assert np.array_equal(got, (np.array([6, 1, 3, 1, 3, 2], np.float64) / U).astype(np.float32))
    # sums: U minus the all-NaN units of each system
    assert [round(float(got[0]) * U), round(float(got[1:4].sum()) * U), round(float(got[4:].sum()) * U)] == [6, 5, 5]


def test_oracle_one_trio_and_uniform_counts():
    rng = np.random.default_rng(0)
    t = rng.uniform(4, 12, (12, 7)).astype(np.float32)
    assert np.array_equal(catalogue_first_trio(t, [1] * 12), np.ones(12, np.float32))
    t[3, 2] = NAN
    assert catalogue_first_trio(t, [1] * 12)[3] == np.float32(6 / 7)
    f = catalogue_first_trio(t, [3] * 4).reshape(4, 3)
    ref = np.zeros((4, 3))
    for n in range(4):
        blk = t[3 * n:3 * n + 3]
        for u in range(7):
            ref[n, np.nanargmin(blk[:, u])] += 1
    assert np.array_equal(f, (ref / 7).astype(np.float32))
    assert np.array_equal(catalogue_first_trio(np.full((2, 3), 5.0, np.float32), [2]), np.array([1, 0], np.float32))


def test_python_argument_errors_before_device_work():
    t = torch.zeros((6, 5))   # a CPU tensor: any device work would raise BnnChaosError, not ValueError
    for counts in ([1, 2], [[3, 3]], [3, 0, 3], [2.0, 4.0], [], [6, 0]):
        with pytest.raises(ValueError):
            first_trio(t, counts)
    for n_trios in (0, -1, 4, 1025):
        with pytest.raises(ValueError):
            first_trio(t, n_trios)
    for bad in (torch.zeros(6), torch.zeros((6, 5, 2))):
        with pytest.raises(ValueError, match="must be"):
            first_trio(bad, 3)
    with pytest.raises(ValueError, match="no units"):
        first_trio(torch.zeros((6, 0)), [3, 3])
    big = torch.zeros((MAX_TRIOS_PER_SYSTEM + 2, 1))
    with pytest.raises(ValueError, match="at most 1024"):
        first_trio(big, [1, MAX_TRIOS_PER_SYSTEM + 1])
    with pytest.raises(_lib.BnnChaosError):   # valid arguments, CPU tensor: no fallback
        first_trio(t, [3, 3])
    with pytest.raises(_lib.BnnChaosError):
        first_trio(t, 3)
    assert MAX_TRIOS_PER_SYSTEM == 1024
    assert check_trio_counts(3, 6) is None and check_trio_counts([1, 1024], None).tolist() == [0, 1, 1025]
    assert check_trio_counts(1024, None) is None


def bare_ensemble():
    """A MultiSWAG without any state: any device work in the method under test would fail with AttributeError."""
    return object.__new__(MultiSWAG)


@pytest.mark.parametrize("rows,kw,match", [
    (6, dict(n_trios=[1, 2]), "sum to 3"),
    (6, dict(n_trios=[3, 0, 3]), "at least one"),
    (6, dict(n_trios=[3, 3], system_offset=2), "system_offset"),
    (6, dict(n_trios=4), "multiple"),
    (1026, dict(n_trios=[1, 1025]), "at most 1024"),
    (1025, dict(n_trios=1025), "at most 1024"),
])
def test_multiswag_trio_errors_before_device_work(rows, kw, match):
    x = torch.zeros((rows, 1, 41))
    with pytest.raises(ValueError, match=match):
        bare_ensemble().posterior_trios(x, 3, **kw)
    if "system_offset" not in kw and match != "sum to 3":   # the sharded form checks a shard's rows on the device
        n_total = len(kw["n_trios"]) if isinstance(kw["n_trios"], list) else rows // kw["n_trios"]
        with pytest.raises(ValueError, match=match):
            bare_ensemble().posterior_trios_sharded(x, n_total, 3, kw["n_trios"])


def test_c_entry_argument_errors():
    """BNN_E_ARG / BNN_E_ALIGN come back before the device is queried; the fake device addresses are never
    dereferenced."""
    lib = _lib.load()
    tp, op, fp = 1 << 20, 3 << 20, 4 << 20
    for args in ((None, 4, 3, 10, fp), (tp, 4, 3, 10, None), (tp, 0, 3, 10, fp), (tp, -1, 3, 10, fp), (tp, 4, 0, 10, fp),
                 (tp, 4, -2, 10, fp), (tp, 4, 1025, 10, fp), (tp, 4, 3, 0, fp), (tp, 4, 3, -3, fp),
                 (tp, 1 << 31, 3, 10, fp), (tp, 4, 3, 1 << 32, fp)):
        assert lib.bnn_first_trio_instability(*args, None) == -1, args   # BNN_E_ARG
        assert lib.bnn_last_error_string().startswith(b"bnn_first_trio_instability:")
    assert lib.bnn_first_trio_instability(tp, 4, 1025, 10, fp, None) == -1
    assert b"1024" in lib.bnn_last_error_string()
    for args in ((tp + 2, 4, 3, 10, fp), (tp, 4, 3, 10, fp + 1)):
        assert lib.bnn_first_trio_instability(*args, None) == -4, args   # BNN_E_ALIGN
        assert b"aligned" in lib.bnn_last_error_string()
    for args in ((None, 4, op, 10, fp), (tp, 4, None, 10, fp), (tp, 4, op, 10, None), (tp, 0, op, 10, fp),
                 (tp, -1, op, 10, fp), (tp, 4, op, 0, fp), (tp, 4, op, -3, fp), (tp, 1 << 31, op, 10, fp),
                 (tp, 4, op, 1 << 32, fp)):
        assert lib.bnn_first_trio_instability_ragged(*args, None) == -1, args   # BNN_E_ARG
        assert lib.bnn_last_error_string().startswith(b"bnn_first_trio_instability_ragged")
    for args in ((tp + 2, 4, op, 10, fp), (tp, 4, op, 10, fp + 1), (tp, 4, op + 4, 10, fp)):
        assert lib.bnn_first_trio_instability_ragged(*args, None) == -4, args   # BNN_E_ALIGN
        assert b"aligned" in lib.bnn_last_error_string()


def test_predict_cli_trios_flag():
    ap = predict.build_parser()
    assert not ap.parse_args(["--models", "m.pkl", "--out", "o"]).trios
    a = ap.parse_args(["--models", "m.pkl", "--data", "c.npz", "--trios", "--survival", "9", "--out", "o"])
    assert a.trios and a.survival == [9.0] and not a.uncertainty
    with pytest.raises(SystemExit):
        ap.parse_args(["--models", "m.pkl", "--out", "o", "--trios", "yes"])


def test_predict_cli_trios_input_validation(tmp_path):
    """More than 1024 trios in a system fails with ValueError before any device work, only with --trios."""
    np.savez(tmp_path / "big.npz", n_trios=[2, 1025], x=np.zeros((1027, 1, 41), np.float32))
    with pytest.raises(ValueError, match="at most 1024"):
        predict.main(["--models", "m.pkl", "--data", str(tmp_path / "big.npz"), "--trios", "--out", str(tmp_path / "o")])
    np.savez(tmp_path / "bad.npz", n_trios=[3, 2], x=np.zeros((6, 1, 41), np.float32))
    with pytest.raises(ValueError):
        predict.main(["--models", "m.pkl", "--data", str(tmp_path / "bad.npz"), "--trios", "--out", str(tmp_path / "o")])
    assert not (tmp_path / "o").exists()


def test_weakest_trio_position():
    counts = np.array([1, 3, 2, 3, 3, 2])
    first = np.array([1.0,
                      0.2, 0.5, 0.3,
                      0.5, 0.5,          # a tie: the first position
                      0.6, 0.2, 0.2,
                      0.1, 0.1, 0.8,
                      0.0, 1.0], np.float32)
    assert predict.weakest_trio_position(first, counts) == {"2": [1, 1], "3": [1, 1, 1]}
    assert predict.weakest_trio_position(np.ones(3, np.float32), np.array([1, 1, 1])) == {}

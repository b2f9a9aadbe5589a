"""CPU: catalogues of mixed planet counts -- the validation of per-system trio counts, catalogue_shard_range, the argument
checks of the ragged C entries (returned before the device is queried), the catalogue oracle against the uniform one,
and the predict CLI's parsing and input validation (before any device work)."""
import ctypes

import numpy as np
import pytest
import torch

from bnn_chaos_model_b200 import _lib, predict
from bnn_chaos_model_b200.multiswag import MultiSWAG, catalogue_shard_range
from bnn_chaos_model_b200.posterior import is_ragged, row_offsets, summarize_instability, survival
from oracle import restatement as R
from oracle.catalogue import catalogue_stats, catalogue_survival, ragged_min_pred, ragged_min_time
from oracle.survival import survival_fraction

INF, NAN = np.inf, np.nan


def test_row_offsets():
    assert row_offsets([1, 3, 2], 6).tolist() == [0, 1, 4, 6] and row_offsets([1, 3, 2], 6).dtype == np.int64
    assert row_offsets(np.array([5], np.int32), 5).tolist() == [0, 5]
    assert row_offsets(torch.tensor([2, 2]), 4).tolist() == [0, 2, 4]
    assert row_offsets((7, 1), None).tolist() == [0, 7, 8]
    for bad, rows, match in (([[1, 2]], 3, "1-D"), ([], 0, "empty"), (np.array([1.0, 2.0]), 3, "integers"),
                             ([True, True], 2, "integers"), ([1, 0, 2], 3, "at least one"), ([2, -1, 2], 3, "at least one"),
                             ([1, 2], 4, "sum to 3"), (torch.tensor([1.5]), 1, "integers")):
        with pytest.raises(ValueError, match=match):
            row_offsets(bad, rows)


def test_is_ragged():
    assert not is_ragged(3) and not is_ragged(np.int64(2)) and not is_ragged(np.array(4)) and not is_ragged(torch.tensor(2))
    assert is_ragged([1, 2]) and is_ragged((3,)) and is_ragged(np.array([1])) and is_ragged(torch.tensor([2, 1]))


def test_posterior_count_errors_before_device_work():
    t, pred = torch.zeros((6, 5)), torch.zeros((6, 5, 2))
    for counts in ([1, 2], [[3, 3]], [3, 0, 3], [2.0, 4.0], []):
        with pytest.raises(ValueError):
            summarize_instability(t, pred, counts)
        with pytest.raises(ValueError):
            survival(t, [9.0], counts)
    with pytest.raises(ValueError):
        survival(t, [NAN], [3, 3])
    with pytest.raises(_lib.BnnChaosError):   # CPU tensors: no fallback
        summarize_instability(t, pred, [3, 3])


def bare_ensemble():
    """A MultiSWAG without any state: any device work in the method under test would fail with AttributeError."""
    return object.__new__(MultiSWAG)


@pytest.mark.parametrize("kw,match", [
    (dict(n_trios=[1, 2]), "sum to 3"),
    (dict(n_trios=[3, 0, 3]), "at least one"),
    (dict(n_trios=[3, 3], system_offset=2), "system_offset"),
])
def test_multiswag_catalogue_errors_before_device_work(kw, match):
    x = torch.zeros((6, 100, 41))
    with pytest.raises(ValueError, match=match):
        bare_ensemble().posterior_summary(x, 3, **kw)
    with pytest.raises(ValueError, match=match):
        bare_ensemble().posterior_survival(x, [9.0], 3, **kw)
    with pytest.raises(ValueError, match=match):
        bare_ensemble().posterior_uncertainty(x, 3, **kw)


def test_catalogue_with_labels_is_refused():
    with pytest.raises(ValueError, match="one trio per system"):
        bare_ensemble()._reduce(torch.zeros((3, 100, 41)), 3, [1, 2], y=torch.zeros((2, 2)))


@pytest.mark.parametrize("seed", range(6))
@pytest.mark.parametrize("g", [1, 5])
def test_catalogue_shard_range(seed, g):
    rng = np.random.default_rng(seed)
    N = [1, 2, 7, 40, 333, 1000][seed]
    counts = rng.integers(1, 9, N)
    off = row_offsets(counts, None)
    Rt = int(off[-1])
    for world in (1, 2, 3, 4, 8, N + 3):
        shards = [catalogue_shard_range(counts, r, world, g) for r in range(world)]
        assert shards[0][0] == 0 and shards[-1][1] == N
        for (slo, shi, rlo, rhi), nxt in zip(shards, shards[1:] + [None]):
            assert slo <= shi and (nxt is None or nxt[0] == shi)   # every system exactly once, in rank order
            assert rlo % g == 0 and (rhi % g == 0 or rhi == Rt)    # the slice is aligned to the granule
            assert rlo <= rhi <= Rt
            if shi > slo:
                assert rlo <= off[slo] < rlo + g and off[shi] <= rhi < off[shi] + g or rhi == Rt
                assert rlo <= off[slo] and off[shi] <= rhi         # owned rows lie inside the slice
            else:
                assert rlo == rhi
        owned = np.array([off[b] - off[a] for a, b, _, _ in shards])
        assert owned.sum() == Rt
        assert (np.abs(owned - Rt / world) <= counts.max()).all(), (world, owned)   # balanced within one system's rows
    assert catalogue_shard_range([3] * 10, 1, 2, 5) == (5, 10, 15, 30)


def test_ragged_entry_argument_errors():
    """BNN_E_ARG / BNN_E_ALIGN come back before the device is queried; the fake device addresses are never
    dereferenced."""
    lib = _lib.load()
    tp, pp, op, sp = 1 << 20, 2 << 20, 3 << 20, 4 << 20
    for args in ((None, pp, 4, op, 10, sp), (tp, None, 4, op, 10, sp), (tp, pp, 4, None, 10, sp), (tp, pp, 4, op, 10, None),
                 (tp, pp, 0, op, 10, sp), (tp, pp, -1, op, 10, sp), (tp, pp, 4, op, 0, sp), (tp, pp, 4, op, -3, sp),
                 (tp, pp, 1 << 31, op, 10, sp)):
        assert lib.bnn_summarize_instability_ragged(*args, None) == -1, args   # BNN_E_ARG
        assert lib.bnn_last_error_string().startswith(b"bnn_summarize_instability_ragged")
    assert lib.bnn_summarize_instability_ragged(tp, pp, 4, op + 4, 10, sp, None) == -4   # BNN_E_ALIGN
    assert b"aligned" in lib.bnn_last_error_string()
    thr = (ctypes.c_float * 3)(4.0, 9.0, NAN)
    for args in ((None, 4, op, 10, thr, 2, sp), (tp, 4, None, 10, thr, 2, sp), (tp, 4, op, 10, None, 2, sp),
                 (tp, 4, op, 10, thr, 2, None), (tp, 0, op, 10, thr, 2, sp), (tp, -1, op, 10, thr, 2, sp),
                 (tp, 4, op, 0, thr, 2, sp), (tp, 4, op, -3, thr, 2, sp), (tp, 4, op, 10, thr, 0, sp),
                 (tp, 4, op, 10, thr, 65, sp), (tp, 1 << 31, op, 10, thr, 2, sp), (tp, 4, op, 1 << 32, thr, 2, sp),
                 (tp, 4, op, 10, thr, 3, sp)):   # the third threshold is NaN
        assert lib.bnn_survival_instability_ragged(*args, None) == -1, args   # BNN_E_ARG
        assert lib.bnn_last_error_string().startswith(b"bnn_survival_instability_ragged")
    assert b"NaN" in lib.bnn_last_error_string()
    for args in ((tp + 2, 4, op, 10, thr, 2, sp), (tp, 4, op, 10, thr, 2, sp + 1), (tp, 4, op + 4, 10, thr, 2, sp)):
        assert lib.bnn_survival_instability_ragged(*args, None) == -4, args   # BNN_E_ALIGN
        assert b"aligned" in lib.bnn_last_error_string()


@pytest.mark.parametrize("Rt", [1, 3])
def test_oracle_equal_counts_match_the_uniform_oracle(Rt):
    rng = np.random.default_rng(Rt)
    N, U = 9, 101
    t = rng.uniform(4, 12, (N * Rt, U)).astype(np.float32)
    pred = np.stack([rng.uniform(4, 12, (N * Rt, U)), rng.uniform(0.5, 6, (N * Rt, U))], -1).astype(np.float32)
    got = catalogue_stats(t, pred, [Rt] * N)
    ref = R.posterior_stats(t.reshape(N, Rt, U).transpose(2, 0, 1), pred.reshape(N, Rt, U, 2).transpose(2, 0, 1, 3))
    for k in ref:
        assert np.array_equal(got[k], ref[k]), k
    thr = [-INF, 5.0, 9.0, INF]
    assert np.array_equal(catalogue_survival(t, thr, [Rt] * N), survival_fraction(t, thr, Rt))


def test_oracle_ragged_min():
    # counts [1, 3, 2]; one unit.  System 1: t (NaN, 5, 7) -> 5; mu (NaN, 6, 4) -> the first trio's NaN is kept (never
    # replaced: nothing is smaller than NaN) and ranks as +inf.  System 2: t all NaN -> +inf; mu (8, 8) -> the first.
    t = np.array([[4.5], [NAN], [5.0], [7.0], [NAN], [NAN]], np.float32)
    mu = np.array([[4.0], [NAN], [6.0], [4.0], [8.0], [8.0]], np.float32)
    sd = np.array([[1.0], [2.0], [3.0], [4.0], [5.0], [6.0]], np.float32)
    counts = [1, 3, 2]
    assert ragged_min_time(t, counts)[:, 0].tolist() == [4.5, 5.0, INF]
    m, s = ragged_min_pred(np.stack([mu, sd], -1), counts)
    assert m[:, 0].tolist() == [4.0, INF, 8.0] and s[:, 0].tolist() == [1.0, 2.0, 5.0]
    mu[1] = 9.0
    m, s = ragged_min_pred(np.stack([mu, sd], -1), counts)
    assert m[:, 0].tolist() == [4.0, 4.0, 8.0] and s[:, 0].tolist() == [1.0, 4.0, 5.0]
    assert catalogue_survival(t, [4.9, 6.0], counts).tolist() == [[0.0, 0.0], [1.0, 0.0], [1.0, 1.0]]


def test_predict_cli_parsing():
    ap = predict.build_parser()
    a = ap.parse_args(["--models", "a.pkl", "b.pkl", "--out", "o"])
    assert a.models == ["a.pkl", "b.pkl"] and a.data is None and a.synthetic == 1000 and a.survival is None
    assert not a.uncertainty and a.samples == 100
    a = ap.parse_args(["--models", "m.pkl", "--data", "c.npz", "--survival", "6", "9", "--uncertainty", "--out", "o"])
    assert a.data == "c.npz" and a.survival == [6.0, 9.0] and a.uncertainty
    for bad in (["--survival"], ["--synthetic", "x"], ["--out"]):
        with pytest.raises(SystemExit):
            ap.parse_args(["--models", "m.pkl", "--out", "o"] + bad)


def test_predict_cli_synthetic_catalogue():
    a = predict.build_parser().parse_args(["--models", "m.pkl", "--synthetic", "50", "--out", "o"])
    counts, inputs = predict.load_catalogue(a)
    assert counts.shape == (50,) and counts.min() >= 1 and counts.max() <= 5 and len(np.unique(counts)) > 2
    assert inputs["x"].shape == (counts.sum(), 100, 41) and inputs["x"].dtype == np.float32
    assert np.array_equal(predict.load_catalogue(a)[0], counts)   # fixed seed


def test_predict_cli_input_validation(tmp_path):
    """Malformed catalogues and bad thresholds fail with ValueError before any device work."""
    x = np.zeros((6, 100, 41), np.float32)
    ts, ms = np.zeros((6, 100, 26)), np.zeros((6, 3))
    cases = {"both": dict(n_trios=[3, 3], x=x, tseries=ts, masses=ms), "neither": dict(n_trios=[3, 3]),
             "sum": dict(n_trios=[3, 2], x=x), "zero": dict(n_trios=[6, 0], x=x), "float": dict(n_trios=[3.0, 3.0], x=x),
             "nocounts": dict(x=x), "nomasses": dict(n_trios=[3, 3], tseries=ts), "shape": dict(n_trios=[3, 3], x=x[..., :40]),
             "rawsum": dict(n_trios=[2, 2], tseries=ts, masses=ms)}
    for name, arrays in cases.items():
        np.savez(tmp_path / f"{name}.npz", **arrays)
        with pytest.raises(ValueError):
            predict.main(["--models", "m.pkl", "--data", str(tmp_path / f"{name}.npz"), "--out", str(tmp_path / "o")])
    np.savez(tmp_path / "ok.npz", n_trios=[3, 3], x=x)
    for bad in (["nan"], [str(v) for v in range(65)]):
        with pytest.raises(ValueError):
            predict.main(["--models", "m.pkl", "--data", str(tmp_path / "ok.npz"), "--out", str(tmp_path / "o"),
                          "--survival"] + bad)
    with pytest.raises(ValueError):
        predict.main(["--models", "m.pkl", "--synthetic", "0", "--out", str(tmp_path / "o")])
    assert not (tmp_path / "o").exists()

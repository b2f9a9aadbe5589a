"""CPU: posterior attribution -- the oracle's float64 reduction and its autograd against the restatement's forward, the
Python argument checks (before any device work), the C entry's argument, shape and alignment errors (returned before
the device is queried) and the predict CLI's --attribution flag."""
import numpy as np
import pytest
import torch

from conftest import swag_stats
from bnn_chaos_model_b200 import _lib, predict, synth
from bnn_chaos_model_b200.multiswag import MultiSWAG
from oracle import restatement as R
from oracle.attribution import reduce_attribution, unit_gradients


def test_oracle_reduction():
    rng = np.random.default_rng(0)
    U, rows, T, F = 3, 4, 5, 6
    g = rng.normal(size=(U, rows, T, F)).astype(np.float32)
    mu = rng.uniform(4, 12, (U, rows)).astype(np.float32)
    attr, mm, abs_shift = reduce_attribution(g, mu)
    assert attr.shape == (rows, 2, F) and mm.shape == (rows,) and abs_shift.shape == (rows, F)
    for r in range(rows):
        for c in range(F):
            v = [[float(g[u, r, t, c]) for t in range(T)] for u in range(U)]
            assert attr[r, 0, c] == pytest.approx(sum(sum(a * a for a in vu) / T for vu in v) / U, rel=1e-14)
            assert attr[r, 1, c] == pytest.approx(sum(sum(vu) for vu in v) / U, rel=1e-12, abs=1e-15)
            assert abs_shift[r, c] == pytest.approx(sum(sum(abs(a) for a in vu) for vu in v) / U, rel=1e-14)
        assert mm[r] == pytest.approx(float(np.mean(mu[:, r].astype(np.float64))), rel=1e-15)
    # shift is signed, importance is not: flipping g keeps importance and negates shift
    a2, _, _ = reduce_attribution(-g, mu)
    assert np.array_equal(a2[:, 0], attr[:, 0]) and np.array_equal(a2[:, 1], -attr[:, 1])


def test_oracle_gradients_match_the_forward():
    """mu of the oracle is forward_swag_fast's mu, and its gradient matches a central difference in one input."""
    st = swag_stats(0)
    spec = R.ModelSpec.from_hparams(st["hparams"])
    x = synth.make_systems(3, seed=4)
    eps = R.draw_eps(2, np.arange(2), np.arange(3), 40)
    thetas = np.stack([st["w_avg"], st["w_avg"] * np.float32(1.01)])
    g, mu = unit_gradients(spec, thetas, x, eps)
    assert g.shape == (2, 3, 100, 41) and mu.shape == (2, 3)
    for u in range(2):
        ref = R.forward_swag_fast(spec, torch.from_numpy(thetas[u]), torch.from_numpy(x), torch.from_numpy(eps[u, :, :20]),
                                  torch.from_numpy(eps[u, :, 20:]))
        np.testing.assert_allclose(mu[u], ref[:, 0].numpy(), rtol=1e-6)
    live = [c for c in range(41) if c not in spec.zero_cols]
    c, t, h = live[2], 40, 1e-2
    spec64 = spec
    th = torch.from_numpy(thetas[0]).double()
    e = torch.from_numpy(eps[0]).double()

    def mu_at(delta):
        xx = torch.from_numpy(x).double().clone()
        xx[0, t, c] += delta
        return float(R.forward_swag_fast(spec64, th, xx, e[:, :20], e[:, 20:])[0, 0])

    fd = (mu_at(h) - mu_at(-h)) / (2 * h)
    assert g[0, 0, t, c] == pytest.approx(fd, rel=2e-2, abs=1e-6)


def bare_ensemble():
    """A MultiSWAG without any state: any device work in the method under test would fail with AttributeError."""
    return object.__new__(MultiSWAG)


@pytest.mark.parametrize("shape,kw,match", [
    ((6, 100, 41), dict(n_trios=[1, 2]), "sum to 3"),
    ((6, 100, 41), dict(n_trios=[3, 0, 3]), "at least one"),
    ((6, 100, 41), dict(n_trios=[3, 3], system_offset=2), "system_offset"),
    ((6, 100, 41), dict(n_trios=4), "multiple"),
    ((6, 100, 41), dict(n_trios=0), "multiple"),
    ((6, 50, 41), dict(), r"\[rows, 100, 41\]"),
    ((6, 100, 40), dict(), r"\[rows, 100, 41\]"),
    ((6, 100), dict(), r"\[N\*n_trios, T, F\]"),
    ((6, 100, 41), dict(max_block_bytes=0), "max_block_bytes"),
    ((6, 100, 41), dict(unit_chunk=0), "unit_chunk"),
])
def test_multiswag_attribution_errors_before_device_work(shape, kw, match):
    x = torch.zeros(shape)
    with pytest.raises(ValueError, match=match):
        bare_ensemble().posterior_attribution(x, 3, **kw)
    with pytest.raises(ValueError, match="samples_per_model"):
        bare_ensemble().posterior_attribution(torch.zeros((6, 100, 41)), 0)


def test_sharded_attribution_errors_before_device_work():
    x = torch.zeros((6, 100, 41))
    with pytest.raises(ValueError, match="trio counts"):
        bare_ensemble().posterior_attribution_sharded(x, 3, 3, [3, 3])
    with pytest.raises(ValueError, match="owns rows"):
        bare_ensemble().posterior_attribution_sharded(x, 3, 3, 1)
    with pytest.raises(ValueError, match="multiple"):
        bare_ensemble().posterior_attribution_sharded(x, 2, 3, 4)


def test_c_entry_argument_errors():
    """BNN_E_ARG / BNN_E_CONFIG / BNN_E_ALIGN come back before the device is queried; the fake device addresses are
    never dereferenced."""
    lib = _lib.load()
    cfg = _lib.ModelConfig(41, 40, 20, 1, 1, 100, 0, 4.0, 12.0, 0.5, 6.0)
    th, xp, ac, at, mm, mu, ws = (k << 20 for k in range(1, 8))
    good = dict(n=4, th=th, u0=0, x=xp, rows=10, r0=0, seed=1, acc=ac, first=1, fin=4, attr=at, mm=mm, mu=mu, ws=ws)

    def call(cfg_=cfg, **kw):
        a = {**good, **kw}
        return lib.bnn_posterior_saliency(cfg_, a["n"], a["th"], a["u0"], a["x"], a["rows"], a["r0"], a["seed"], a["acc"],
                                          a["first"], a["fin"], a["attr"], a["mm"], a["mu"], a["ws"], None)

    for kw in (dict(th=None), dict(x=None), dict(acc=None), dict(ws=None), dict(attr=None), dict(mm=None), dict(n=0),
               dict(n=65536), dict(rows=0), dict(rows=1 << 30), dict(u0=-1), dict(r0=-1), dict(u0=(1 << 32) - 3),
               dict(r0=(1 << 32) - 9), dict(fin=-1), dict(fin=3), dict(fin=1 << 32)):
        assert call(**kw) == -1, kw   # BNN_E_ARG
        assert lib.bnn_last_error_string().startswith(b"bnn_posterior_saliency"), kw
    for t, f in ((52, 41), (100, 40)):
        bad = _lib.ModelConfig(f, 40, 20, 1, 1, t, 0, 4.0, 12.0, 0.5, 6.0)
        assert call(bad) == -2, (t, f)   # BNN_E_CONFIG
        assert b"T=100, F=41" in lib.bnn_last_error_string()
    assert call(None) == -1
    for kw in (dict(ws=ws + 8), dict(acc=ac + 4), dict(x=xp + 2), dict(th=th + 1), dict(attr=at + 2), dict(mm=mm + 1),
               dict(mu=mu + 3)):
        assert call(**kw) == -4, kw   # BNN_E_ALIGN
        assert b"aligned" in lib.bnn_last_error_string()
    assert lib.bnn_posterior_saliency_workspace_bytes(cfg, 0, 10) == 0
    assert lib.bnn_posterior_saliency_workspace_bytes(cfg, 4, 0) == 0
    n = lib.bnn_posterior_saliency_workspace_bytes(cfg, 148, 440)
    assert n > 148 * 440 * (100 * 41 + 40 + 1) * 4 + 148 * 440 * 83 * 8   # gradients, draws, mu, double partial sums


def test_workspace_query_is_monotone():
    """A workspace sized for (n_units, rows) serves every smaller call: the query never shrinks when either count grows,
    although the saliency kernel's CTA count per call (SMs / n_units, capped by the system pairs) is not monotone."""
    lib = _lib.load()
    cfg = _lib.ModelConfig(41, 40, 20, 1, 1, 100, 0, 4.0, 12.0, 0.5, 6.0)
    ws = lambda n, r: lib.bnn_posterior_saliency_workspace_bytes(cfg, n, r)
    units = list(range(1, 200)) + [296, 1000, 65535]
    rows = [1, 2, 3, 5, 31, 40, 50, 200, 442]
    for r in rows:
        sizes = [ws(n, r) for n in units]
        assert all(a <= b for a, b in zip(sizes, sizes[1:])), r
    for n in (1, 9, 10, 74, 100, 148, 149):
        sizes = [ws(n, r) for r in rows]
        assert all(a <= b for a, b in zip(sizes, sizes[1:])), n
    assert ws(10, 31) >= ws(9, 31) > 0 and ws(100, 40) >= ws(74, 40)


def test_predict_cli_attribution_flag(tmp_path):
    ap = predict.build_parser()
    assert not ap.parse_args(["--models", "m.pkl", "--out", "o"]).attribution
    a = ap.parse_args(["--models", "m.pkl", "--data", "c.npz", "--attribution", "--trios", "--out", "o"])
    assert a.attribution and a.trios and not a.uncertainty
    with pytest.raises(SystemExit):
        ap.parse_args(["--models", "m.pkl", "--out", "o", "--attribution", "yes"])
    np.savez(tmp_path / "short.npz", n_trios=[1, 2], x=np.zeros((3, 50, 41), np.float32))
    with pytest.raises(ValueError, match="T = 100"):
        predict.main(["--models", "m.pkl", "--data", str(tmp_path / "short.npz"), "--attribution", "--out",
                      str(tmp_path / "o")])
    assert not (tmp_path / "o").exists()

"""GPU: the short N-body integration (K8, bnn_integrate_orbits) against oracle/nbody.py for P = 3..8, on encounter
cases, against scipy's DOP853 (second-order convergence), energy over 10^4 orbits, bit-identity of a system alone, in a
batch and in a mixed catalogue, the C entry's argument errors, a weak in-distribution pack check, and predict on an
orbit catalogue (one process and 2 ranks, and the refusal of an ensemble that reads columns 1-7)."""
import json
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT, make_swag_model, swag_stats
from test_gpu_catalogue import free_port, save_models
from bnn_chaos_model_b200 import _lib, nbody, predict, synth
from bnn_chaos_model_b200.inputs import data_setup_kernel
from oracle import nbody as O

pytestmark = pytest.mark.gpu

ENERGY_BOUND = 1e-6   # |dE / E| over 10^3 - 10^4 orbits; the oracle's worst over 8 systems at 10^3 orbits is 4e-8


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


def angle_diff(a, b):
    return np.abs(O.wrap(a - b + np.pi) - np.pi)


def compare_rows(got, ref, rel=1e-9, ang=1e-9):
    assert np.array_equal(np.isnan(got), np.isnan(ref))
    g, r = np.nan_to_num(got), np.nan_to_num(ref)
    assert np.array_equal(g[..., :8], r[..., :8])
    for j in range(3):
        b = 8 + 6 * j
        err = np.abs(g[..., b:b + 3] - r[..., b:b + 3]) / np.maximum(np.abs(r[..., b:b + 3]), 1e-300)
        small = np.abs(r[..., b + 1:b + 3]) < 1e-6   # e, inc near 0: absolute
        err[..., 1:][small] = np.abs(g[..., b + 1:b + 3] - r[..., b + 1:b + 3])[small]
        assert err.max() <= rel, (j, err.max())
        assert angle_diff(g[..., b + 3:b + 6], r[..., b + 3:b + 6]).max() <= ang


@pytest.mark.parametrize("P", [3, 4, 5, 6, 7, 8])
def test_device_matches_oracle(dev, P):
    el = synth.initial_orbits(4, P, seed=40 + P, spacing=(10.0, 20.0))
    ts, ms, lt = nbody.integrate_orbits(el, P, n_orbits=100, device=dev)
    rts, rms, rlt = O.integrate(el, n_orbits=100)
    assert np.array_equal(ms.cpu().numpy(), rms)
    assert np.isnan(lt.cpu().numpy()).all() and np.isnan(rlt).all()
    compare_rows(ts.cpu().numpy(), rts)


def crossing_systems(n, seed):
    """3-planet systems whose middle planet's orbit crosses the inner one's: clear-cut encounters."""
    rng = np.random.default_rng(seed)
    el = synth.initial_orbits(n, 3, seed=seed, spacing=(10.0, 14.0))
    el[:, 1, 2] = rng.uniform(0.3, 0.5, n)
    el[:, :, 0] = 3e-5
    return el


def test_encounter_step_matches_oracle(dev):
    el = crossing_systems(12, 5)
    ts, _, lt = nbody.integrate_orbits(el, 3, n_orbits=100, device=dev)
    rts, _, rlt, sep = O.integrate(el, n_orbits=100, trace=True)
    lt, ts = lt.cpu().numpy(), ts.cpu().numpy()
    hit = np.isfinite(rlt)
    assert hit.sum() >= 3
    for n in np.flatnonzero(hit):
        s = int(np.flatnonzero(sep[:, n] < 1.0)[0]) if (sep[:, n] < 1.0).any() else None
        if s is not None and not (0.999 < sep[s, n] < 1.001) and (s == 0 or sep[s - 1, n] > 1.001):
            assert abs(lt[n] - rlt[n]) <= 1e-12, n
            assert np.array_equal(np.isnan(ts[n]), np.isnan(rts[n]))
    # crossing orbits that survive are chaotic: rounding differences grow, so only their NaN pattern must agree
    assert np.isnan(lt[~hit]).all() and not np.isnan(ts[~hit]).any()


def test_dop853_second_order_on_device(dev):
    for P in (3, 5):
        el = synth.initial_orbits(1, P, seed=P, spacing=(12.0, 16.0), e_max=0.08)
        errs = []
        for f in (0.05, 0.025, 0.0125):
            ts, _, _ = nbody.integrate_orbits(el, P, n_orbits=20, dt_frac=f, device=dev)
            ts = ts.cpu().numpy()
            _, P1 = O.timestep(el, f)
            rows = np.arange(80, 100)
            ref = O.newtonian_reference(el[0], ts[0, rows, 0] * P1[0])
            g = np.empty((rows.size, P, 6))
            for p in range(P):
                i = min(p, P - 3)
                g[:, p] = ts[i][rows][:, 8 + 6 * (p - i):14 + 6 * (p - i)]
                g[:, p, 0] *= el[0, i, 1]
            d = np.abs(g - ref)
            d[..., 5] = angle_diff(g[..., 5], ref[..., 5])
            errs.append(d[..., [0, 1, 2, 5]].max())
        r = np.array(errs[:-1]) / np.array(errs[1:])
        assert ((r > 3.0) & (r < 5.0)).all(), (P, errs)


def test_energy_over_1e4_orbits(dev):
    el = synth.initial_orbits(64, 3, seed=8, spacing=(12.0, 20.0))
    ts, ms, lt = nbody.integrate_orbits(el, 3, device=dev)
    ts, ms, lt = ts.cpu().numpy(), ms.cpu().numpy(), lt.cpu().numpy()
    E0 = O.energy(el)
    ok = np.isnan(lt)
    assert ok.sum() >= 32
    for n in np.flatnonzero(ok):
        E = O.energy_from_rows(ts[n][[0, -1]], ms[n], el[n, 0, 1])
        assert np.abs((E - E0[n]) / E0[n]).max() < ENERGY_BOUND


def test_bits_independent_of_batch(dev):
    one = synth.initial_orbits(1, 5, seed=77)
    batch = synth.initial_orbits(10000, 5, seed=78)
    batch[5000] = one[0]
    counts = np.array([3, 8, 5, 4, 6, 7, 5, 3])
    mixed = synth.initial_orbits(counts.size, counts, seed=79)
    off = np.concatenate([[0], np.cumsum(counts)])
    mixed[off[2]:off[3]] = one[0]
    a = nbody.integrate_orbits(one, 5, n_orbits=100, device=dev)
    b = nbody.integrate_orbits(batch, 5, n_orbits=100, device=dev)
    c = nbody.integrate_orbits(mixed, counts, n_orbits=100, device=dev)
    roff = np.concatenate([[0], np.cumsum(counts - 2)])
    assert torch.equal(a[0], b[0][15000:15003]) and torch.equal(a[0], c[0][roff[2]:roff[3]])
    assert torch.equal(a[1], b[1][15000:15003]) and torch.equal(a[1], c[1][roff[2]:roff[3]])
    assert torch.equal(a[2].isnan(), b[2][5000:5001].isnan())
    # every system of the mixed catalogue equals its own launch
    for n, P in enumerate(counts):
        s = nbody.integrate_orbits(mixed[off[n]:off[n + 1]], int(P), n_orbits=100, device=dev)
        assert torch.equal(s[0], c[0][roff[n]:roff[n + 1]])


def test_c_entry_argument_errors(dev):
    lib = _lib.load()
    el = torch.from_numpy(synth.initial_orbits(2, 3, seed=1)).to(dev)
    ts = torch.full((2, 100, 26), 7.0, dtype=torch.float64, device=dev)
    ms = torch.full((2, 3), 7.0, dtype=torch.float64, device=dev)
    lt = torch.full((2,), 7.0, dtype=torch.float64, device=dev)
    p = lambda t: t.data_ptr()
    good = [p(el), 2, 3, 100.0, 0.05, p(ts), p(ms), p(lt), None]
    cases = [(0, None), (5, None), (6, None), (7, None), (1, 0), (1, 1 << 31), (2, 2), (2, 9), (3, 0.0), (3, float("nan")),
             (3, float("inf")), (4, -1.0), (4, float("nan")), (3, 1e9)]
    for i, v in cases:
        args = list(good)
        args[i] = v
        assert lib.bnn_integrate_orbits(*args) == -1, (i, v)
    for i in (0, 5, 6, 7):
        args = list(good)
        args[i] = args[i] + 4
        assert lib.bnn_integrate_orbits(*args) == -4, i
    torch.cuda.synchronize()
    assert (ts == 7.0).all() and (ms == 7.0).all() and (lt == 7.0).all()
    assert lib.bnn_integrate_orbits(*good) == 0


def test_invalid_elements_give_nan_rows(dev):
    lib = _lib.load()
    el = synth.initial_orbits(4, 3, seed=2, spacing=(14.0, 20.0))
    el[1, 1, 1] = -1.0
    el[2, 0, 2] = 1.0
    el[3, 2, 5] = np.nan
    d = torch.from_numpy(el).to(dev)
    ts = torch.empty((4, 100, 26), dtype=torch.float64, device=dev)
    ms = torch.empty((4, 3), dtype=torch.float64, device=dev)
    lt = torch.empty(4, dtype=torch.float64, device=dev)
    assert lib.bnn_integrate_orbits(d.data_ptr(), 4, 3, 10.0, 0.05, ts.data_ptr(), ms.data_ptr(), lt.data_ptr(), None) == 0
    ts, lt = ts.cpu().numpy(), lt.cpu().numpy()
    assert not np.isnan(ts[0]).any() and np.isnan(ts[1:]).all() and np.isnan(lt).all()


def test_pack_in_distribution_weak(dev):
    """WEAK in-distribution check: synth.initial_orbits systems that survive 10^4 orbits pack to finite standardised
    live columns, and at least 98 % of them stay within +-6 (the v50 scaler's units) at every output.  The rest are
    planets scattered by a close approach that stops short of Hill-sphere overlap (the instability test): a light planet
    that loses a few % of its a is many scaler units out, since column 8's scale is 0.0047.  The check shows only that
    the conventions land in the training range."""
    el = synth.initial_orbits(256, 3, seed=11)
    ts, ms, lt = nbody.integrate_orbits(el, 3, device=dev)
    x = data_setup_kernel(ms, ts)
    ok = torch.isnan(lt)   # survived the integration
    live = [0] + list(range(8, 38))
    z = x[ok][:, :, live]
    assert ok.sum() > 128 and z.isfinite().all()
    inside = (z.abs() < 6.0).flatten(1).all(1)
    assert inside.float().mean() >= 0.98


def orbit_catalogue(tmp_path, n=30, seed=5):
    counts = np.random.default_rng(seed).integers(3, 9, n)
    el = synth.initial_orbits(n, counts, seed=seed, spacing=(4.0, 14.0))
    path = str(tmp_path / "orbits.npz")
    np.savez(path, orbits=el, n_planets=counts)
    return path, el, counts


def test_predict_orbit_catalogue_matches_tseries(dev, tmp_path):
    paths = save_models(tmp_path, dev, (0, 3))
    cat, el, counts = orbit_catalogue(tmp_path)
    extra = ["--samples", "3", "--survival", "5", "9", "--uncertainty", "--trios", "--attribution"]
    predict.main(["--models", *paths, "--data", cat, "--n_orbits", "1000", "--out", str(tmp_path / "o")] + extra)
    ts, ms, lt = nbody.integrate_orbits(el, counts, n_orbits=1000, device=dev)
    raw = str(tmp_path / "raw.npz")
    np.savez(raw, tseries=ts.cpu().numpy(), masses=ms.cpu().numpy(), n_trios=counts - 2)
    predict.main(["--models", *paths, "--data", raw, "--out", str(tmp_path / "r")] + extra)
    zo, zr = np.load(tmp_path / "o" / "per_system.npz"), np.load(tmp_path / "r" / "per_system.npz")
    lt = lt.cpu().numpy()
    assert np.array_equal(zo["log10_t_unstable"], lt, equal_nan=True) and np.isfinite(lt).any()
    want = nbody.override_unstable(dict(zr), lt, counts - 2)
    assert sorted(zo.files) == sorted(list(zr.files) + ["log10_t_unstable"])
    for k in zr.files:
        if zr[k].dtype.kind in "fc":
            assert np.array_equal(zo[k], want[k], equal_nan=True), k
        else:
            assert np.array_equal(zo[k], want[k]), k
    hit = np.isfinite(lt)
    assert (zo["summary"][hit, :6] == lt[hit, None].astype(np.float32)).all() and np.isnan(zo["summary"][hit, 6:]).all()
    info = json.load(open(tmp_path / "o" / "summary.json"))
    assert info["n_unstable_in_integration"] == int(hit.sum()) and info["n_orbits"] == 1000.0 and info["dt_frac"] == 0.05


def test_predict_orbit_catalogue_under_torchrun_world2(dev, tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    paths = save_models(tmp_path, dev, (0, 3))
    cat, _, _ = orbit_catalogue(tmp_path, n=41, seed=6)
    common = ["--models", *paths, "--data", cat, "--n_orbits", "500", "--samples", "3", "--survival", "9",
              "--uncertainty", "--trios", "--attribution"]
    predict.main(common + ["--out", str(tmp_path / "one")])
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", "2", "--master-port", str(free_port()),
           "-m", "bnn_chaos_model_b200.predict"] + common + ["--out", str(tmp_path / "two")]
    p = subprocess.run(cmd, cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, timeout=900)
    assert p.returncode == 0, p.stdout.decode()[-4000:]
    z1, z2 = np.load(tmp_path / "one" / "per_system.npz"), np.load(tmp_path / "two" / "per_system.npz")
    assert sorted(z1.files) == sorted(z2.files)
    for k in z1.files:
        assert np.array_equal(z1[k], z2[k], equal_nan=z1[k].dtype.kind == "f"), k


def test_predict_refuses_ensemble_reading_mmr(dev, tmp_path):
    from bnn_chaos_model_b200 import spock_reg_model as S

    st = swag_stats(0)
    m = S.SWAGModel(dict(st["hparams"], include_mmr=True)).init_params(st["swa_params"]).to(dev)
    m.w_avg, m.w2_avg, m.pre_D = (torch.from_numpy(st[k]).to(dev) for k in ("w_avg", "w2_avg", "pre_D"))
    path = str(tmp_path / "mmr_output.pkl")
    S.save_swag(m, path)
    cat, _, _ = orbit_catalogue(tmp_path, n=4)
    with pytest.raises(ValueError, match=r"columns \[3, 6\]"):
        predict.main(["--models", path, "--data", cat, "--n_orbits", "10", "--out", str(tmp_path / "x")])

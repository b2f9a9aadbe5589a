"""CPU: the short N-body integration's restatement (oracle/nbody.py) against physics that does not rest on our code
(exact Kepler motion of massless planets, scipy's DOP853 on the inertial Newtonian ODE, energy), its encounter test,
the output grid and row layout, and every ValueError of nbody.integrate_orbits, nbody.override_unstable and predict's
orbit catalogue loader."""
import argparse

import numpy as np
import pytest

from bnn_chaos_model_b200 import nbody, predict, synth
from oracle import nbody as O

# |dE / E| over 10^3 orbits.  Wisdom-Holman without a corrector has a bounded energy error of order
# max(m) (n dt)^2 ~ 5e-5 (2 pi 0.05)^2 ~ 5e-6 at worst; the oracle's largest over the 8 systems below is 4e-8.
ENERGY_BOUND = 1e-6


def angle_diff(a, b):
    return np.abs(O.wrap(a - b + np.pi) - np.pi)


def test_massless_planets_are_exact_kepler():
    el = synth.initial_orbits(3, 3, seed=1, spacing=(10.0, 20.0), e_max=0.1)
    el[:, :, 0] = 0.0
    ts, _, lt = O.integrate(el, n_orbits=100)
    assert np.isnan(lt).all()
    for n in range(3):
        for j in range(3):
            blk = ts[n][:, 8 + 6 * j:14 + 6 * j]
            assert np.abs(blk[:, :3] - blk[0, :3]).max() < 1e-12
            assert angle_diff(blk[:, 3:5], blk[0, 3:5]).max() < 1e-11 / max(el[n, j, 2], 1e-3)
            lam = O.rows_to_elements(ts[n], el[n, 0, 1])[:, j, 5]
            a = el[n, j, 1]
            t = ts[n][:, 0] * O.TWO_PI          # P1 = 2 pi for a1 = 1 about M = 1
            assert angle_diff(lam, el[n, j, 6] + t * a ** -1.5).max() < 1e-9


@pytest.mark.parametrize("P", [3, 5])
def test_second_order_against_dop853(P):
    el = synth.initial_orbits(1, P, seed=P, spacing=(12.0, 16.0), e_max=0.08)
    errs = []
    for f in (0.05, 0.025, 0.0125):
        ts, _, _ = O.integrate(el, n_orbits=20, dt_frac=f)
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
    assert ((r > 3.0) & (r < 5.0)).all(), errs


def test_energy_over_1e3_orbits():
    el = synth.initial_orbits(8, 3, seed=1, spacing=(10.0, 20.0))
    ts, ms, lt = O.integrate(el, n_orbits=1000)
    assert np.isnan(lt).all()
    E0 = O.energy(el)
    for n in range(8):
        E = O.energy_from_rows(ts[n][[0, -1]], ms[n], el[n, 0, 1])
        assert abs((E[0] - E0[n]) / E0[n]) < 1e-14
        assert abs((E[1] - E0[n]) / E0[n]) < ENERGY_BOUND


def test_encounter_flagged_at_first_overlap():
    el = synth.initial_orbits(6, 3, seed=5, spacing=(10.0, 14.0))
    el[:, 1, 2] = np.random.default_rng(5).uniform(0.3, 0.5, 6)
    el[:, :, 0] = 3e-5
    ts, _, lt, sep = O.integrate(el, n_orbits=100, trace=True)
    dt, P1 = O.timestep(el, 0.05)
    steps = O.output_steps(100, dt, P1)
    hit = np.flatnonzero(np.isfinite(lt))
    assert hit.size >= 2
    for n in hit:
        s = int(np.flatnonzero(sep[:, n] < 1.0)[0]) + 1       # trace row s - 1 is step s's kick
        assert s == 1 or sep[s - 2, n] >= 1.0                  # not at the step before
        assert np.isnan(sep[s:, n]).all()                      # the system stopped there
        assert lt[n] == np.log10(s * dt[n] / P1[n])
        k = int(np.searchsorted(steps[n], s))                  # first output at or after the step: NaN from there
        assert np.isnan(ts[n][k:]).all() and not np.isnan(ts[n][:k]).any()


def test_grid_layout_and_trio_normalisation():
    el = synth.initial_orbits(2, 5, seed=3, spacing=(12.0, 20.0))
    ts, ms, lt = O.integrate(el, n_orbits=30)
    dt, P1 = O.timestep(el, 0.05)
    assert ts.shape == (6, 100, 26) and ms.shape == (6, 3) and np.isnan(lt).all()
    for n in range(2):
        t = ts[3 * n][:, 0]
        want = O.output_steps(30, dt[n], P1[n]) * dt[n] / P1[n]
        assert np.array_equal(t, want) and t[0] == 0.0
        grid = 10 * np.arange(100) * 30 / 999
        assert (t >= grid - 1e-12).all() and (t - dt[n] / P1[n] < grid).all()
        for i in range(3):
            r = ts[3 * n + i]
            assert np.array_equal(r[:, 0], t) and (r[:, 1:8] == 0).all()
            assert np.array_equal(ms[3 * n + i], el[n, i:i + 3, 0])
            assert abs(r[0, 8] - 1.0) < 1e-12                                  # a / a_{i,0} of the trio's inner planet
            assert np.allclose(r[0, 8::6], el[n, i:i + 3, 1] / el[n, i, 1], rtol=1e-12)
            assert ((r[:, [11, 12, 13, 17, 18, 19, 23, 24, 25]] >= 0) & (r[:, [11, 12, 13, 17, 18, 19, 23, 24, 25]]
                                                                            < 2 * np.pi)).all()
        # a planet shared by trios has the same elements in each (up to its normalisation)
        assert np.array_equal(ts[3 * n][:, 15:20], ts[3 * n + 1][:, 9:14])


def test_invalid_systems_are_nan():
    el = synth.initial_orbits(3, 3, seed=2, spacing=(14.0, 20.0))
    el[1, 0, 2] = 1.0
    ts, ms, lt = O.integrate(el, n_orbits=5)
    assert np.isnan(ts[1]).all() and not np.isnan(ts[0]).any() and np.isnan(lt).all()
    assert np.array_equal(ms[1], el[1, :, 0])


def test_integrate_orbits_value_errors():
    el = synth.initial_orbits(2, 4, seed=1)
    flat = el.reshape(-1, 7)
    bad = [(flat, 2), (flat, 9), (flat, 3), (flat, np.array([4, 3])), (flat, np.array([4, 5])), (flat, np.array([2, 6])),
           (flat, np.array([4.0, 4.0])), (flat[:, :6], 4)]
    for e, n in bad:
        with pytest.raises(ValueError):
            nbody.integrate_orbits(e, n)
    for col, v, msg in [(1, 0.0, "a <= 0"), (2, 1.0, "e outside"), (2, -0.1, "e outside"), (0, -1e-6, "negative mass"),
                        (4, np.nan, "non-finite"), (1, 0.5, "increase")]:
        x = flat.copy()
        x[1, col] = v
        with pytest.raises(ValueError, match=msg):
            nbody.integrate_orbits(x, 4)
    for kw in ({"n_orbits": 0.0}, {"n_orbits": np.inf}, {"dt_frac": -1.0}, {"dt_frac": np.nan}, {"n_orbits": 1e9}):
        with pytest.raises(ValueError):
            nbody.integrate_orbits(flat, 4, **kw)


def test_override_unstable():
    counts = np.array([1, 3, 2])
    rng = np.random.default_rng(0)
    arrays = {"summary": rng.random((3, 8)).astype(np.float32), "survival": rng.random((3, 2)).astype(np.float32),
              "thresholds": np.array([5.0, 9.0], np.float32), "uncertainty": rng.random((6, 5)).astype(np.float32),
              "trio_first": rng.random(6).astype(np.float32), "attribution": rng.random((6, 2, 41)).astype(np.float32),
              "n_trios": counts}
    lt = np.array([np.nan, 6.5, np.nan])
    out = nbody.override_unstable(arrays, lt, counts)
    assert np.array_equal(out["summary"][[0, 2]], arrays["summary"][[0, 2]])
    assert (out["summary"][1, :6] == np.float32(6.5)).all() and np.isnan(out["summary"][1, 6:]).all()
    assert np.array_equal(out["survival"][1], [1.0, 0.0]) and np.array_equal(out["survival"][[0, 2]], arrays["survival"][[0, 2]])
    for k in ("uncertainty", "trio_first", "attribution"):
        assert np.isnan(out[k][1:4]).all() and np.array_equal(out[k][[0, 4, 5]], arrays[k][[0, 4, 5]])
    assert out["n_trios"] is counts and not np.isnan(arrays["summary"]).any()
    with pytest.raises(ValueError):
        nbody.override_unstable(arrays, lt[:2], counts)
    with pytest.raises(ValueError):
        nbody.override_unstable({k: v for k, v in arrays.items() if k != "thresholds"}, lt, counts)
    with pytest.raises(ValueError):
        nbody.override_unstable(dict(arrays, uncertainty=arrays["uncertainty"][:5]), lt, counts)
    with pytest.raises(ValueError):
        nbody.override_unstable(dict(arrays, summary=arrays["summary"][:2]), lt, counts)
    with pytest.raises(ValueError):
        nbody.override_unstable(arrays, lt, np.array([1, 3, 0]))


def test_orbit_catalogue_loader(tmp_path):
    counts = np.array([3, 5, 4])
    el = synth.initial_orbits(3, counts, seed=4)
    ok = tmp_path / "ok.npz"
    np.savez(ok, orbits=el, n_planets=counts)
    n_trios, inputs = predict.load_catalogue(argparse.Namespace(data=str(ok)))
    assert np.array_equal(n_trios, counts - 2) and np.array_equal(inputs["orbits"], el)
    bad_el = el.copy()
    bad_el[4, 2] = 1.5
    cases = {"both": dict(orbits=el, n_planets=counts, x=np.zeros((9, 100, 41), np.float32)),
             "no_counts": dict(orbits=el), "no_orbits": dict(n_planets=counts),
             "shape": dict(orbits=el[:, :6], n_planets=counts), "sum": dict(orbits=el, n_planets=np.array([3, 5, 5])),
             "range": dict(orbits=el, n_planets=np.array([2, 6, 4])), "values": dict(orbits=bad_el, n_planets=counts),
             "trios": dict(orbits=el, n_planets=counts, n_trios=counts)}
    for name, z in cases.items():
        p = tmp_path / f"{name}.npz"
        np.savez(p, **z)
        with pytest.raises(ValueError):
            predict.load_catalogue(argparse.Namespace(data=str(p)))

"""Synthetic 3-planet orbital time series with the model's input shape [N, 100, 41].

There is no network and the reference's training data is not in its repository
(/root/reference/data/README.md), so benchmarks and parity tests run on generated
systems.  The generator follows the column convention of the reference's input
builder (figures/spock/regression.py:183-213 ``data_setup_kernel``): 26 time-series
columns + 3 masses + 3 nan flags, with the nine angle columns
{11,12,13,17,18,19,23,24,25} expanded to (cos, sin) -> 41 columns, then the
StandardScaler constants hard-coded in ``load_swag`` (spock_reg_model.py:934-955).
Values are chosen so that the v50 checkpoints give in-distribution predictions
(median mu ~ 5.7, a few % saturated at the soft clamps).
"""
from __future__ import annotations

import numpy as np

# spock_reg_model.py:934-955 (v50 fixed scaler; identical to figures/spock/regression.py:48-70)
SSX_SCALE = np.array([
    2.88976974e+03, 6.10019661e-02, 4.03849732e-02, 4.81638693e+01, 6.72583662e-02, 4.17939679e-02,
    8.15995339e+00, 2.26871589e+01, 4.73612029e-03, 7.09223721e-02, 3.06455099e-02, 7.10726478e-01,
    7.03392022e-01, 7.07873597e-01, 7.06030923e-01, 7.04728204e-01, 7.09420909e-01, 1.90740659e-01,
    4.75502285e-02, 2.77188320e-02, 7.08891412e-01, 7.05214134e-01, 7.09786887e-01, 7.04371833e-01,
    7.04371110e-01, 7.09828420e-01, 3.33589977e-01, 5.20857790e-02, 2.84763136e-02, 7.02210626e-01,
    7.11815232e-01, 7.10512240e-01, 7.03646004e-01, 7.08017286e-01, 7.06162814e-01, 2.12569430e-05,
    2.35019125e-05, 2.04211110e-05, 7.51048890e-02, 3.94254400e-01, 7.11351099e-02])
SSX_MEAN = np.array([
    4.95458585e+03, 5.67411891e-02, 3.83176945e-02, 2.97223474e+00, 6.29733979e-02, 3.50074471e-02,
    6.72845676e-01, 9.92794768e+00, 9.99628430e-01, 5.39591547e-02, 2.92795061e-02, 2.12480714e-03,
    -1.01500319e-02, 1.82667162e-02, 1.00813201e-02, 5.74404197e-03, 6.86570242e-03, 1.25316320e+00,
    4.76946516e-02, 2.71326280e-02, 7.02054326e-03, 9.83378673e-03, -5.70616748e-03, 5.50782881e-03,
    -8.44213953e-04, 2.05958338e-03, 1.57866569e+00, 4.31476211e-02, 2.73316392e-02, 1.05505555e-02,
    1.03922250e-02, 7.36865006e-03, -6.00523246e-04, 6.53016990e-03, -1.72038113e-03, 1.24807860e-05,
    1.60314173e-05, 1.21732696e-05, 5.67292645e-03, 1.92488263e-01, 5.08607199e-03])

ANGLE_COLS = (11, 12, 13, 17, 18, 19, 23, 24, 25)  # figures/spock/regression.py:200
N_RAW, N_FEATURES, N_TIMES = 32, 41, 100


def raw_systems(n: int, seed: int = 0, t: int = N_TIMES) -> np.ndarray:
    """Raw (un-normalised, angles not yet expanded) series, float64 [n, t, 32]."""
    rng = np.random.default_rng(seed)
    time = np.linspace(0.0, 1e4, t)[None, :]
    X = np.zeros((n, t, N_RAW))
    X[:, :, 0] = time
    # columns 1..7 (e+-, mmr strength, megno): arbitrary plausible values; the v50 flags zero them
    X[:, :, 1:8] = SSX_MEAN[1:8] + 0.3 * SSX_SCALE[1:8] * rng.standard_normal((n, t, 7))
    a = np.ones((n, 3))
    a[:, 1] = a[:, 0] + rng.uniform(0.05, 0.5, n)
    a[:, 2] = a[:, 1] + rng.uniform(0.05, 0.6, n)
    for j in range(3):
        base = 8 + 6 * j
        X[:, :, base + 0] = a[:, j, None] * (1.0 + 1e-3 * rng.standard_normal((n, t)))
        e0 = rng.uniform(0.0, 0.1, (n, 1))
        per = rng.uniform(500.0, 5000.0, (n, 1))
        X[:, :, base + 1] = np.abs(e0 + 0.01 * np.sin(2 * np.pi * time / per))
        X[:, :, base + 2] = rng.uniform(0.0, 0.06, (n, 1)) * np.ones((1, t))
        X[:, :, base + 3] = rng.uniform(0, 2 * np.pi, (n, 1)) - 2 * np.pi * time / rng.uniform(2e3, 2e4, (n, 1))
        X[:, :, base + 4] = rng.uniform(0, 2 * np.pi, (n, 1)) + 2 * np.pi * time / rng.uniform(2e3, 2e4, (n, 1))
        X[:, :, base + 5] = rng.uniform(0, 2 * np.pi, (n, 1)) + 2 * np.pi * time * a[:, j, None] ** -1.5 * 1.0137
    X[:, :, 26:29] = (10.0 ** rng.uniform(-7.0, -4.3, (n, 3)))[:, None, :]
    # nan flags (29..31) stay 0
    return X


def expand_angles(raw: np.ndarray) -> np.ndarray:
    """[.., 32] -> [.., 41]: cos/sin expansion of the angle columns (regression.py:198-207)."""
    cols = []
    for j in range(raw.shape[-1]):
        if j in ANGLE_COLS:
            cols.append(np.cos(raw[..., [j]]))
            cols.append(np.sin(raw[..., [j]]))
        else:
            cols.append(raw[..., [j]])
    return np.concatenate(cols, axis=-1)


def standardize(X41: np.ndarray) -> np.ndarray:
    """sklearn StandardScaler.transform in float64, as the callers do before .float()."""
    return (X41 - SSX_MEAN) / SSX_SCALE


def make_systems(n: int, seed: int = 0, t: int = N_TIMES, normalised: bool = True) -> np.ndarray:
    """fp32 [n, t, 41] model inputs (normalised by default, like every caller passes them)."""
    X = expand_angles(raw_systems(n, seed, t))
    if normalised:
        X = standardize(X)
    return np.ascontiguousarray(X, dtype=np.float32)


def make_labels(n: int, seed: int = 0) -> np.ndarray:
    """fp32 [n, 2] log10 instability times; >= 9 is the censored ('stable') branch."""
    rng = np.random.default_rng(seed + 7919)
    return rng.uniform(4.0, 10.0, (n, 2)).astype(np.float32)


def initial_orbits(n: int, n_planets, seed: int = 0, spacing=(5.0, 20.0), e_max: float = 0.05,
                   inc_max: float = 0.05) -> np.ndarray:
    """Initial orbits for ``nbody.integrate_orbits``: [n, P, 7] for an int ``n_planets``, or [sum P, 7] for per-system
    counts [n].  Per planet (m, a, e, inc, Omega, varpi, lambda): m = 10^U(-7, -4.3) (the masses of ``raw_systems``),
    a1 = 1 and each next a spaced U(spacing) mutual Hill radii out, e ~ U(0, e_max), inc ~ U(0, inc_max), angles
    U(0, 2 pi).  Systems in the range the v50 ensembles were trained on, some of them unstable within 10^4 orbits; of
    those that survive, a few (under 2 % of 3-planet systems) have a planet scattered out of that range by a close
    approach that stops short of Hill-sphere overlap."""
    rng = np.random.default_rng(seed)
    counts = np.full(n, int(n_planets)) if np.ndim(n_planets) == 0 else np.asarray(n_planets, dtype=np.int64)
    if counts.size != n:
        raise ValueError(f"{counts.size} planet counts for {n} systems")
    el = np.empty((int(counts.sum()), 7))
    el[:, 0] = 10.0 ** rng.uniform(-7.0, -4.3, el.shape[0])
    el[:, 2] = rng.uniform(0.0, e_max, el.shape[0])
    el[:, 3] = rng.uniform(0.0, inc_max, el.shape[0])
    el[:, 4:7] = rng.uniform(0.0, 2 * np.pi, (el.shape[0], 3))
    delta = rng.uniform(spacing[0], spacing[1], el.shape[0])
    first = np.concatenate([[0], np.cumsum(counts)[:-1]])
    # a_{p+1} = a_p (1 + k) / (1 - k), k = delta ((m_p + m_{p+1}) / 3)^(1/3) / 2: the planets delta mutual Hill radii apart
    k = delta[1:] * ((el[:-1, 0] + el[1:, 0]) / 3.0) ** (1.0 / 3.0) / 2.0
    log_ratio = np.concatenate([[0.0], np.log((1.0 + k) / (1.0 - k))])
    log_ratio[first] = 0.0
    cum = np.cumsum(log_ratio)
    el[:, 1] = np.exp(cum - np.repeat(cum[first], counts))
    return el.reshape(n, int(n_planets), 7) if np.ndim(n_planets) == 0 else el

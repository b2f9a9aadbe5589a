"""Plain-numpy fp64 restatement of the short N-body integration (csrc/nbody.cu, ``bnn_integrate_orbits``).

Same element conversion, same step order, same Newton rule and same encounter test as the kernel, vectorised over
systems of one planet count P.  G = 1, M_star = 1; each planet is (m, a, e, inc, Omega, varpi, lambda) in Jacobi
elements, planets ordered from the inside out.  The kernel contracts a*b + c into FMA where numpy rounds twice, so the
two agree to rounding, not bit for bit.
"""
from __future__ import annotations

import numpy as np

TWO_PI = 2.0 * np.pi
N_OUT = 100            # output rows per trio
N_COLS = 26            # raw time-series columns per row
KEPLER_TOL = 1e-12     # Newton in the eccentric-anomaly increment stops after the first update with |dx| < KEPLER_TOL
KEPLER_CAP = 30        # ... or after KEPLER_CAP updates
ROT_SMALL = 0.05       # |dx| below this: sin / cos of the update from a degree-8 Taylor polynomial, else sincos


def wrap(a):
    """Angle in [0, 2 pi)."""
    w = np.fmod(a, TWO_PI)
    w = np.where(w < 0.0, w + TWO_PI, w)
    return np.where(w >= TWO_PI, 0.0, w)


def output_times(n_orbits: float, P1):
    """t_k = 10 k n_orbits / 999 P1, k = 0..99 (P1: the innermost planet's initial period)."""
    k = np.arange(N_OUT, dtype=np.float64)
    return (10.0 * k) * n_orbits / 999.0 * np.asarray(P1)[..., None]


def _sincos_small(d):
    d2 = d * d
    s = d * (1.0 - d2 / 6.0 * (1.0 - d2 / 20.0 * (1.0 - d2 / 42.0)))
    c = 1.0 - d2 / 2.0 * (1.0 - d2 / 12.0 * (1.0 - d2 / 30.0 * (1.0 - d2 / 56.0)))
    return s, c


def rotate_back(sx, cx, dx):
    """(sin(x - dx), cos(x - dx)) from (sin x, cos x)."""
    small = np.abs(dx) < ROT_SMALL
    sd, cd = _sincos_small(np.where(small, dx, 0.0))
    sd = np.where(small, sd, np.sin(dx))
    cd = np.where(small, cd, np.cos(dx))
    return sx * cd - cx * sd, cx * cd + sx * sd


def elements_to_cartesian(mu, a, e, inc, Om, pom, lam):
    """Jacobi position and velocity (each a tuple of 3 arrays) of an orbit about mass mu."""
    om = pom - Om
    M = wrap(lam - pom)
    E = np.where(e < 0.8, M, np.pi)
    active = np.ones_like(E, dtype=bool)
    for _ in range(KEPLER_CAP):
        dE = (E - e * np.sin(E) - M) / (1.0 - e * np.cos(E))
        E = np.where(active, E - dE, E)
        active &= ~(np.abs(dE) < KEPLER_TOL)
    sE, cE = np.sin(E), np.cos(E)
    q = np.sqrt(1.0 - e * e)
    n = np.sqrt(mu / (a * a * a))
    xp, yp = a * (cE - e), a * q * sE
    vs = n * a / (1.0 - e * cE)
    vxp, vyp = -sE * vs, q * cE * vs
    co, so, cO, sO, ci, si = np.cos(om), np.sin(om), np.cos(Om), np.sin(Om), np.cos(inc), np.sin(inc)
    # R3(Omega) R1(inc) R3(omega)
    r11, r12 = cO * co - sO * so * ci, -cO * so - sO * co * ci
    r21, r22 = sO * co + cO * so * ci, -sO * so + cO * co * ci
    r31, r32 = so * si, co * si
    return ((r11 * xp + r12 * yp, r21 * xp + r22 * yp, r31 * xp + r32 * yp),
            (r11 * vxp + r12 * vyp, r21 * vxp + r22 * vyp, r31 * vxp + r32 * vyp))


def cartesian_to_elements(mu, x, y, z, vx, vy, vz):
    """(a, e, inc, Omega, varpi, theta) of the osculating orbit about mass mu; angles in [0, 2 pi), Omega = 0 for a
    planar orbit."""
    r = np.sqrt(x * x + y * y + z * z)
    v2 = vx * vx + vy * vy + vz * vz
    rv = x * vx + y * vy + z * vz
    hx, hy, hz = y * vz - z * vy, z * vx - x * vz, x * vy - y * vx
    hxy2 = hx * hx + hy * hy
    h = np.sqrt(hxy2 + hz * hz)
    a = 1.0 / (2.0 / r - v2 / mu)
    ecf = h * h / (mu * r) - 1.0
    esf = h * rv / (mu * r)
    e = np.sqrt(ecf * ecf + esf * esf)
    hxy = np.sqrt(hxy2)
    inc = np.arctan2(hxy, hz)
    Om = np.where(hxy2 > 0.0, np.arctan2(hx, -hy), 0.0)
    cO, sO = np.cos(Om), np.sin(Om)
    ci, si = hz / h, hxy / h
    u = np.arctan2(-x * ci * sO + y * ci * cO + z * si, x * cO + y * sO)
    f = np.arctan2(esf, ecf)
    th = Om + u
    return a, e, inc, wrap(Om), wrap(th - f), wrap(th)


def kepler_drift(mu, x, y, z, vx, vy, vz, h):
    """Advance every Jacobi orbit by h (Gauss f and g in the eccentric-anomaly increment).  Returns the new state and
    `bound`: False where 2/r - v^2/mu <= 0 (or NaN), where the state is returned unchanged."""
    r0 = np.sqrt(x * x + y * y + z * z)
    v2 = vx * vx + vy * vy + vz * vz
    rv = x * vx + y * vy + z * vz
    alpha = 2.0 / r0 - v2 / mu
    bound = alpha > 0.0
    alpha = np.where(bound, alpha, 1.0)
    a = 1.0 / alpha
    n = np.sqrt(mu * alpha * alpha * alpha)
    c = 1.0 - r0 * alpha
    s = rv / (n * a * a)
    X = n * h
    sx, cx = np.sin(X), np.cos(X)
    active = np.ones_like(X, dtype=bool)
    for _ in range(KEPLER_CAP):
        fp = 1.0 - c * cx + s * sx
        dx = (X - c * sx + s * (1.0 - cx) - n * h) / fp
        dx = np.where(active, dx, 0.0)
        X = X - dx
        sx, cx = rotate_back(sx, cx, dx)
        active &= ~(np.abs(dx) < KEPLER_TOL)
    rr = a * (1.0 - c * cx + s * sx)
    f = 1.0 - (1.0 - cx) / (r0 * alpha)
    g = h - (X - sx) / n
    fd = -(n * a * a) * sx / (rr * r0)
    gd = 1.0 - a * (1.0 - cx) / rr
    nx, ny, nz = f * x + g * vx, f * y + g * vy, f * z + g * vz
    nvx, nvy, nvz = fd * x + gd * vx, fd * y + gd * vy, fd * z + gd * vz
    keep = lambda new, old: np.where(bound, new, old)
    return (keep(nx, x), keep(ny, y), keep(nz, z), keep(nvx, vx), keep(nvy, vy), keep(nvz, vz)), bound


def interior_masses(m):
    """M_i = 1 + m_1 + .. + m_i, summed from the star outwards (the Jacobi Kepler mass of planet i)."""
    M = np.empty_like(m)
    acc = np.ones(m.shape[:-1])
    for i in range(m.shape[-1]):
        acc = acc + m[..., i]
        M[..., i] = acc
    return M


def valid_systems(el):
    """Per system: every planet has finite values, m >= 0, a > 0 and 0 <= e < 1."""
    fin = np.isfinite(el).all(-1)
    ok = fin & (el[..., 0] >= 0.0) & (el[..., 1] > 0.0) & (el[..., 2] >= 0.0) & (el[..., 2] < 1.0)
    return ok.all(-1)


def timestep(el, dt_frac):
    """(dt, P1): dt = dt_frac min_i P_i (1 - e_i)^(3/2) / sqrt(1 + e_i), P_i = 2 pi sqrt(a_i^3 / M_i)."""
    m, a, e = el[..., 0], el[..., 1], el[..., 2]
    per = TWO_PI * np.sqrt(a * a * a / interior_masses(m))
    w = per * ((1.0 - e) * np.sqrt(1.0 - e) / np.sqrt(1.0 + e))
    return dt_frac * w.min(-1), per[..., 0]


def output_steps(n_orbits, dt, P1):
    """Step index of each output: the first step boundary s dt >= t_k."""
    return np.ceil(output_times(n_orbits, P1) / np.asarray(dt)[..., None])


def jacobi_state(el):
    """Jacobi positions and velocities, 6 arrays [N, P], of the elements [N, P, 7]."""
    mu = interior_masses(el[..., 0])
    r, v = elements_to_cartesian(mu, *(el[..., k] for k in range(1, 7)))
    return list(r) + list(v)


def inertial_positions(m, M, x, y, z):
    """Planet positions [N, P] in the frame of the star (star at the origin), from Jacobi positions."""
    P = m.shape[-1]
    X, Y, Z = np.empty_like(x), np.empty_like(y), np.empty_like(z)
    Rx = Ry = Rz = np.zeros(m.shape[:-1])
    for i in range(P):
        X[:, i], Y[:, i], Z[:, i] = Rx + x[:, i], Ry + y[:, i], Rz + z[:, i]
        q = m[:, i] / M[:, i]
        Rx, Ry, Rz = Rx + q * x[:, i], Ry + q * y[:, i], Rz + q * z[:, i]
    return X, Y, Z


def kick(m, M, hill, s, h):
    """Jacobi interaction kick of length h on the state s (6 arrays [N, P], changed in place).  Returns (close,
    sep): close where two planets are nearer than the sum of their Hill radii, sep the smallest |d| / (h_j + h_k)."""
    x, y, z, vx, vy, vz = s
    N, P = m.shape
    X, Y, Z = inertial_positions(m, M, x, y, z)
    # inertial accelerations by direct summation over all pairs, the star (mass 1, at the origin) included
    ax, ay, az = np.zeros((N, P)), np.zeros((N, P)), np.zeros((N, P))
    a0x, a0y, a0z = np.zeros(N), np.zeros(N), np.zeros(N)
    close = np.zeros(N, bool)
    sep = np.full(N, np.inf)
    for j in range(P):
        r2 = X[:, j] * X[:, j] + Y[:, j] * Y[:, j] + Z[:, j] * Z[:, j]
        ir3 = 1.0 / (r2 * np.sqrt(r2))
        ax[:, j] -= X[:, j] * ir3
        ay[:, j] -= Y[:, j] * ir3
        az[:, j] -= Z[:, j] * ir3
        a0x += m[:, j] * X[:, j] * ir3
        a0y += m[:, j] * Y[:, j] * ir3
        a0z += m[:, j] * Z[:, j] * ir3
    for j in range(P):
        for k in range(j + 1, P):
            dx, dy, dz = X[:, k] - X[:, j], Y[:, k] - Y[:, j], Z[:, k] - Z[:, j]
            d2 = dx * dx + dy * dy + dz * dz
            rh = hill[:, j] + hill[:, k]
            close |= d2 < rh * rh
            sep = np.minimum(sep, np.sqrt(d2) / rh)
            ir3 = 1.0 / (d2 * np.sqrt(d2))
            ax[:, j] += m[:, k] * dx * ir3
            ay[:, j] += m[:, k] * dy * ir3
            az[:, j] += m[:, k] * dz * ir3
            ax[:, k] -= m[:, j] * dx * ir3
            ay[:, k] -= m[:, j] * dy * ir3
            az[:, k] -= m[:, j] * dz * ir3
    # to Jacobi (a'_i = a_i - A_{i-1}, A the interior centre of mass's acceleration), minus the Keplerian term
    Ax, Ay, Az = a0x, a0y, a0z
    for i in range(P):
        jx, jy, jz = ax[:, i] - Ax, ay[:, i] - Ay, az[:, i] - Az
        q = m[:, i] / M[:, i]
        Ax, Ay, Az = Ax + q * jx, Ay + q * jy, Az + q * jz
        r2 = x[:, i] * x[:, i] + y[:, i] * y[:, i] + z[:, i] * z[:, i]
        kep = M[:, i] / (r2 * np.sqrt(r2))
        vx[:, i] += h * (jx + kep * x[:, i])
        vy[:, i] += h * (jy + kep * y[:, i])
        vz[:, i] += h * (jz + kep * z[:, i])
    return close, sep


def all_bound(M, s):
    x, y, z, vx, vy, vz = s
    alpha = 2.0 / np.sqrt(x * x + y * y + z * z) - (vx * vx + vy * vy + vz * vz) / M
    return (alpha > 0.0).all(-1)


def drift(M, s, h):
    with np.errstate(all="ignore"):
        out, _ = kepler_drift(M, *s, np.asarray(h)[:, None])
    return [np.array(c) for c in out]


def write_rows(ts, M, s, el, P1, t, due, k):
    """Rows k (per system) of every trio of the systems `due` from the synchronised state s."""
    N, P = M.shape
    with np.errstate(all="ignore"):
        elem = cartesian_to_elements(M, *s)
    nt = P - 2
    for n in np.flatnonzero(due):
        for i in range(nt):
            row = ts[n * nt + i, k[n]]
            row[:] = 0.0
            row[0] = t[n] / P1[n]
            for j in range(3):
                p = i + j
                row[8 + 6 * j] = elem[0][n, p] / el[n, i, 1]
                for c in range(1, 6):
                    row[8 + 6 * j + c] = elem[c][n, p]


def integrate(elements, n_orbits=1e4, dt_frac=0.05, trace=False):
    """elements [N, P, 7] -> (tseries [N (P - 2), 100, 26], masses [N (P - 2), 3], log10_t_unstable [N]) as
    bnn_integrate_orbits writes them; with trace=True also sep [n_steps, N], the smallest |d| / (h_j + h_k) at each
    step's kick (NaN after a system stops)."""
    el = np.array(elements, dtype=np.float64)
    N, P, _ = el.shape
    nt = P - 2
    masses = np.stack([el[:, i:i + 3, 0] for i in range(nt)], 1).reshape(N * nt, 3)
    ts = np.full((N * nt, N_OUT, N_COLS), np.nan)
    lt = np.full(N, np.nan)
    ok = valid_systems(el)
    el_run = np.where(ok[:, None, None], el, np.array([1e-9, 1.0, 0.0, 0.0, 0.0, 0.0, 0.0]) * np.ones((N, P, 7))
                      + np.where(np.arange(7) == 1, np.arange(P)[:, None], 0.0))
    with np.errstate(all="ignore"):
        dt, P1 = timestep(el_run, dt_frac)
        steps = output_steps(n_orbits, dt, P1)
    n_steps = steps[:, -1]
    ok &= n_steps <= 2.0 ** 31
    m = el_run[..., 0]
    M = interior_masses(m)
    hill = el_run[..., 1] * np.cbrt(m / 3.0)
    s = jacobi_state(el_run)
    live = ok.copy()
    kout = np.zeros(N, np.int64)
    due = live & (steps[np.arange(N), np.minimum(kout, N_OUT - 1)] == 0)
    while due.any():
        write_rows(ts, M, s, el, P1, np.zeros(N), due, kout)
        kout += due
        due = live & (kout < N_OUT) & (steps[np.arange(N), np.minimum(kout, N_OUT - 1)] == 0)
    s = drift(M, s, 0.5 * dt)
    sep_trace = []
    total = int(n_steps[ok].max()) if ok.any() else 0
    for step in range(1, total + 1):
        live &= step <= n_steps
        if not live.any():
            break
        old = [c.copy() for c in s]
        with np.errstate(all="ignore"):
            close, sep = kick(m, M, hill, s, dt)
            bad = (close | ~all_bound(M, s)) & live
        if trace:
            sep_trace.append(np.where(live, sep, np.nan))
        lt[bad] = np.log10(step * dt[bad] / P1[bad])
        live &= ~bad
        s = [np.where(live[:, None], c, o) for c, o in zip(s, old)]
        due = live & (kout < N_OUT) & (steps[np.arange(N), np.minimum(kout, N_OUT - 1)] == step)
        if due.any():
            z = drift(M, s, 0.5 * dt)
            while due.any():
                write_rows(ts, M, z, el, P1, step * dt, due, kout)
                kout += due
                due = live & (kout < N_OUT) & (steps[np.arange(N), np.minimum(kout, N_OUT - 1)] == step)
        if step < total:
            s = drift(M, s, dt)
    if trace:
        return ts, masses, lt, np.array(sep_trace)
    return ts, masses, lt


def energy(el):
    """Total energy of the systems [N, P, 7] in their centre-of-mass frame (G = M_star = 1)."""
    m = el[..., 0]
    M = interior_masses(m)
    x, y, z, vx, vy, vz = jacobi_state(el)
    Mprev = np.concatenate([np.ones(m.shape[:-1] + (1,)), M[..., :-1]], -1)
    kin = 0.5 * (m * Mprev / M * (vx * vx + vy * vy + vz * vz)).sum(-1)
    X, Y, Z = inertial_positions(m, M, x, y, z)
    pot = -(m / np.sqrt(X * X + Y * Y + Z * Z)).sum(-1)
    P = m.shape[-1]
    for j in range(P):
        for k in range(j + 1, P):
            pot -= m[:, j] * m[:, k] / np.sqrt((X[:, k] - X[:, j]) ** 2 + (Y[:, k] - Y[:, j]) ** 2 + (Z[:, k] - Z[:, j]) ** 2)
    return kin + pot


def rows_to_elements(rows, a0):
    """Rows [T, 26] of a trio and its innermost initial a -> Jacobi elements (a, e, inc, Omega, varpi, lambda) [T, 3, 6]:
    the mean longitude lambda from theta through the true and eccentric anomalies."""
    out = np.stack([rows[:, 8 + 6 * j:14 + 6 * j] for j in range(3)], 1).copy()
    out[..., 0] *= a0
    e, pom, th = out[..., 1], out[..., 4], out[..., 5]
    f = th - pom
    E = 2.0 * np.arctan2(np.sqrt(1.0 - e) * np.sin(0.5 * f), np.sqrt(1.0 + e) * np.cos(0.5 * f))
    out[..., 5] = wrap(pom + E - e * np.sin(E))
    return out


def energy_from_rows(rows, masses, a0):
    """Energy [T] of a 3-planet system from its single trio's rows [T, 26] and masses [3]."""
    el = rows_to_elements(rows, a0)
    full = np.concatenate([np.broadcast_to(np.asarray(masses, np.float64), el.shape[:2])[..., None], el], -1)
    return energy(full)


def jacobi_to_inertial(m, s):
    """Jacobi state (6 arrays [N, P]) -> centre-of-mass positions and velocities [N, P + 1, 3] of star and planets."""
    M = interior_masses(m)
    w = np.concatenate([np.ones((m.shape[0], 1)), m], 1)

    def com_frame(x, y, z):   # the same linear map takes Jacobi positions and velocities to star-origin ones
        X = np.stack(inertial_positions(m, M, x, y, z), -1)
        allp = np.concatenate([np.zeros(X.shape[:1] + (1, 3)), X], 1)
        return allp - (w[..., None] * allp).sum(1, keepdims=True) / w.sum(1)[:, None, None]

    return com_frame(*s[:3]), com_frame(*s[3:])


def inertial_to_elements(m, pos, vel):
    """Centre-of-mass positions and velocities [N, P + 1, 3] -> Jacobi elements (a, e, inc, Omega, varpi, theta), each
    [N, P]."""
    M = interior_masses(m)
    P = m.shape[1]
    r, v = np.empty(pos.shape[:1] + (P, 3)), np.empty(pos.shape[:1] + (P, 3))
    Rc, Vc, Mprev = pos[:, 0], vel[:, 0], np.ones(m.shape[0])
    for i in range(P):
        r[:, i], v[:, i] = pos[:, i + 1] - Rc, vel[:, i + 1] - Vc
        Rc = (Mprev[:, None] * Rc + m[:, i, None] * pos[:, i + 1]) / M[:, i, None]
        Vc = (Mprev[:, None] * Vc + m[:, i, None] * vel[:, i + 1]) / M[:, i, None]
        Mprev = M[:, i]
    return cartesian_to_elements(M, *(r[..., k] for k in range(3)), *(v[..., k] for k in range(3)))


def newtonian_reference(el, t_eval, rtol=1e-13, atol=1e-13):
    """The inertial Newtonian N-body ODE integrated by scipy's DOP853 from the elements [P, 7] of one system; returns
    the Jacobi elements (a, e, inc, Omega, varpi, theta) [len(t_eval), P] at the times t_eval.  Independent of the
    Wisdom-Holman code: only the element conversions are shared."""
    from scipy.integrate import solve_ivp

    el = np.asarray(el, np.float64)[None]
    m = el[..., 0]
    pos, vel = jacobi_to_inertial(m, jacobi_state(el))
    P = m.shape[1]
    w = np.concatenate([[1.0], m[0]])

    def rhs(_, y):
        p = y[:3 * (P + 1)].reshape(P + 1, 3)
        d = p[None, :, :] - p[:, None, :]
        r3 = (d * d).sum(-1) ** 1.5
        np.fill_diagonal(r3, np.inf)
        acc = (w[None, :, None] * d / r3[..., None]).sum(1)
        return np.concatenate([y[3 * (P + 1):], acc.reshape(-1)])

    y0 = np.concatenate([pos[0].reshape(-1), vel[0].reshape(-1)])
    sol = solve_ivp(rhs, (0.0, float(np.max(t_eval))), y0, method="DOP853", rtol=rtol, atol=atol, t_eval=t_eval)
    Y = sol.y.T
    T = Y.shape[0]
    pos = Y[:, :3 * (P + 1)].reshape(T, P + 1, 3)
    vel = Y[:, 3 * (P + 1):].reshape(T, P + 1, 3)
    return np.stack(inertial_to_elements(np.repeat(m, T, 0), pos, vel), -1)

// K8: the short N-body integration that turns initial orbits into the model's raw time series (bnn_integrate_orbits).
//
// WHFast-style Wisdom-Holman in Jacobi coordinates, fp64, one system per thread, one template instantiation per planet
// count P (3..8) so the state stays in registers.  G = 1, M_star = 1.  Planet i (inside out) is given by the Jacobi
// elements (m, a, e, inc, Omega, varpi, lambda) about the primary "star + planets 1..i-1", with mu_i = M_i = 1 + m_1 +
// .. + m_i.  oracle/nbody.py restates the algorithm in numpy, operation for operation.
//
// Step k (k = 1..n) is drift(dt/2) kick(dt) drift(dt/2); consecutive half drifts are merged, so the integrated state Y
// lives half a step ahead of the step boundaries:
//   Y = D(dt/2) X0;  for k = 1..n:  K(dt) Y  [encounter + unbound test]  [outputs due at k: D(dt/2) of a copy of Y]
//                                    Y = D(dt) Y
// No symplectic corrector.  The kick is the Jacobi interaction term: inertial accelerations by direct summation over
// every pair, the star included, transformed to Jacobi, minus each coordinate's Keplerian term.  The drift is Gauss's
// f and g in the eccentric-anomaly increment x, by Newton from x = n dt with one sincos; later iterates rotate (sin x,
// cos x) by the update (a degree-8 Taylor polynomial below |dx| = 0.05) instead of calling sincos again, and stop after
// the first update with |dx| < 1e-12, or after 30.
//
// Our conventions (SPOCK's setup code is not in this repository, so where the v50 scaler does not pin them they are
// ours): dt = dt_frac min_i P_i (1 - e_i)^(3/2) / sqrt(1 + e_i) (a pericentre rule), outputs at the first step
// boundary t >= t_k = 10 k n_orbits / 999 P1, k = 0..99 (REBOUND's exact_finish_time = 0), one row of 26 doubles per
// adjacent trio (i, i+1, i+2): t / P1, 0 x 7 (e+-, MMR strength and MEGNO are not computed), then per trio planet
// (a / a_{i,0}, e, inc, Omega, varpi, theta = Omega + omega + f), angles in [0, 2 pi).  a_{i,0} is the initial a of the
// trio's innermost planet: a1 for P = 3, and for outer trios the choice that keeps column 8 near 1, as in training.
//
// A system is unstable at the first step whose kick sees two planets nearer than the sum of their Hill radii
// a_{j,0} (m_j / 3)^(1/3), or after whose kick a Jacobi orbit has 2/r - v^2/mu <= 0 (unbound: the elliptic drift
// cannot proceed).  Its thread stops there: the output rows at that step and later are NaN, and log10_t_unstable =
// log10(k dt / P1).  A system that reaches its last output has log10_t_unstable = NaN.
#include <math.h>

#include "common.cuh"

namespace bnn {
namespace {

constexpr int NB_OUT = 100, NB_COLS = 26, NB_THREADS = 128;
constexpr double NB_TWO_PI = 6.283185307179586;  // 2.0 * np.pi
constexpr double NB_KEPLER_TOL = 1e-12;
constexpr int NB_KEPLER_CAP = 30;
constexpr double NB_ROT_SMALL = 0.05;

__device__ __forceinline__ double wrap_angle(double a) {
    double w = fmod(a, NB_TWO_PI);
    if (w < 0.0) w += NB_TWO_PI;
    return w >= NB_TWO_PI ? 0.0 : w;
}

// (sin(x - d), cos(x - d)) from (sin x, cos x)
__device__ __forceinline__ void rotate_back(double& sx, double& cx, double d) {
    double sd, cd;
    if (fabs(d) < NB_ROT_SMALL) {
        const double d2 = d * d;
        sd = d * (1.0 - d2 / 6.0 * (1.0 - d2 / 20.0 * (1.0 - d2 / 42.0)));
        cd = 1.0 - d2 / 2.0 * (1.0 - d2 / 12.0 * (1.0 - d2 / 30.0 * (1.0 - d2 / 56.0)));
    } else {
        sincos(d, &sd, &cd);
    }
    const double s = sx * cd - cx * sd;
    cx = cx * cd + sx * sd;
    sx = s;
}

struct Orbit {
    double x, y, z, vx, vy, vz;
};

// Gauss f and g: advance the Kepler orbit about mu by h.  The caller guarantees 2/r - v^2/mu > 0.
__device__ __forceinline__ void kepler_drift(Orbit& o, double mu, double h) {
    const double r0 = sqrt(o.x * o.x + o.y * o.y + o.z * o.z);
    const double v2 = o.vx * o.vx + o.vy * o.vy + o.vz * o.vz;
    const double rv = o.x * o.vx + o.y * o.vy + o.z * o.vz;
    const double alpha = 2.0 / r0 - v2 / mu;
    const double a = 1.0 / alpha;
    const double n = sqrt(mu * alpha * alpha * alpha);
    const double c = 1.0 - r0 * alpha;
    const double s = rv / (n * a * a);
    double X = n * h, sx, cx;
    sincos(X, &sx, &cx);
    for (int it = 0; it < NB_KEPLER_CAP; ++it) {
        const double fp = 1.0 - c * cx + s * sx;
        const double dx = (X - c * sx + s * (1.0 - cx) - n * h) / fp;
        X = X - dx;
        rotate_back(sx, cx, dx);
        if (fabs(dx) < NB_KEPLER_TOL) break;
    }
    const double rr = a * (1.0 - c * cx + s * sx);
    const double f = 1.0 - (1.0 - cx) / (r0 * alpha);
    const double g = h - (X - sx) / n;
    const double fd = -(n * a * a) * sx / (rr * r0);
    const double gd = 1.0 - a * (1.0 - cx) / rr;
    const Orbit p = o;
    o.x = f * p.x + g * p.vx;
    o.y = f * p.y + g * p.vy;
    o.z = f * p.z + g * p.vz;
    o.vx = fd * p.x + gd * p.vx;
    o.vy = fd * p.y + gd * p.vy;
    o.vz = fd * p.z + gd * p.vz;
}

__device__ __forceinline__ Orbit elements_to_orbit(double mu, double a, double e, double inc, double Om, double pom,
                                                   double lam) {
    const double om = pom - Om;
    const double M = wrap_angle(lam - pom);
    double E = e < 0.8 ? M : 3.141592653589793;
    for (int it = 0; it < NB_KEPLER_CAP; ++it) {
        const double dE = (E - e * sin(E) - M) / (1.0 - e * cos(E));
        E = E - dE;
        if (fabs(dE) < NB_KEPLER_TOL) break;
    }
    double sE, cE, so, co, sO, cO, si, ci;
    sincos(E, &sE, &cE);
    sincos(om, &so, &co);
    sincos(Om, &sO, &cO);
    sincos(inc, &si, &ci);
    const double q = sqrt(1.0 - e * e);
    const double n = sqrt(mu / (a * a * a));
    const double xp = a * (cE - e), yp = a * q * sE;
    const double vs = n * a / (1.0 - e * cE);
    const double vxp = -sE * vs, vyp = q * cE * vs;
    const double r11 = cO * co - sO * so * ci, r12 = -cO * so - sO * co * ci;
    const double r21 = sO * co + cO * so * ci, r22 = -sO * so + cO * co * ci;
    const double r31 = so * si, r32 = co * si;
    return Orbit{r11 * xp + r12 * yp, r21 * xp + r22 * yp, r31 * xp + r32 * yp,
                 r11 * vxp + r12 * vyp, r21 * vxp + r22 * vyp, r31 * vxp + r32 * vyp};
}

// (a, e, inc, Omega, varpi, theta) of the osculating orbit about mu
__device__ __forceinline__ void orbit_to_elements(const Orbit& o, double mu, double* out) {
    const double r = sqrt(o.x * o.x + o.y * o.y + o.z * o.z);
    const double v2 = o.vx * o.vx + o.vy * o.vy + o.vz * o.vz;
    const double rv = o.x * o.vx + o.y * o.vy + o.z * o.vz;
    const double hx = o.y * o.vz - o.z * o.vy, hy = o.z * o.vx - o.x * o.vz, hz = o.x * o.vy - o.y * o.vx;
    const double hxy2 = hx * hx + hy * hy;
    const double h = sqrt(hxy2 + hz * hz);
    const double ecf = h * h / (mu * r) - 1.0;
    const double esf = h * rv / (mu * r);
    const double hxy = sqrt(hxy2);
    const double Om = hxy2 > 0.0 ? atan2(hx, -hy) : 0.0;
    double sO, cO;
    sincos(Om, &sO, &cO);
    const double ci = hz / h, si = hxy / h;
    const double u = atan2(-o.x * ci * sO + o.y * ci * cO + o.z * si, o.x * cO + o.y * sO);
    const double f = atan2(esf, ecf);
    const double th = Om + u;
    out[0] = 1.0 / (2.0 / r - v2 / mu);
    out[1] = sqrt(ecf * ecf + esf * esf);
    out[2] = atan2(hxy, hz);
    out[3] = wrap_angle(Om);
    out[4] = wrap_angle(th - f);
    out[5] = wrap_angle(th);
}

// Per-thread constants live in shared memory, [quantity][planet][thread], so the registers hold the orbits.
template <int P>
struct Consts {
    double* base;
    __device__ double& m(int i) const { return base[(0 * P + i) * NB_THREADS + threadIdx.x]; }
    __device__ double& M(int i) const { return base[(1 * P + i) * NB_THREADS + threadIdx.x]; }
    __device__ double& hill(int i) const { return base[(2 * P + i) * NB_THREADS + threadIdx.x]; }
};

template <int P>
struct System {
    Orbit o[P];
    Consts<P> c;
};

// Kick of length h.  Returns true when two planets are nearer than the sum of their Hill radii at the kick's
// positions, or when a Jacobi orbit is unbound after it.
template <int P>
__device__ __forceinline__ bool kick(System<P>& s, double h) {
    double X[P], Y[P], Z[P], ax[P], ay[P], az[P];
    double Rx = 0.0, Ry = 0.0, Rz = 0.0;
#pragma unroll
    for (int i = 0; i < P; ++i) {
        X[i] = Rx + s.o[i].x;
        Y[i] = Ry + s.o[i].y;
        Z[i] = Rz + s.o[i].z;
        const double q = s.c.m(i) / s.c.M(i);
        Rx = Rx + q * s.o[i].x;
        Ry = Ry + q * s.o[i].y;
        Rz = Rz + q * s.o[i].z;
    }
    double a0x = 0.0, a0y = 0.0, a0z = 0.0;
#pragma unroll
    for (int j = 0; j < P; ++j) {
        const double r2 = X[j] * X[j] + Y[j] * Y[j] + Z[j] * Z[j];
        const double ir3 = 1.0 / (r2 * sqrt(r2));
        ax[j] = -X[j] * ir3;
        ay[j] = -Y[j] * ir3;
        az[j] = -Z[j] * ir3;
        a0x += s.c.m(j) * X[j] * ir3;
        a0y += s.c.m(j) * Y[j] * ir3;
        a0z += s.c.m(j) * Z[j] * ir3;
    }
    bool close = false;
#pragma unroll
    for (int j = 0; j < P; ++j) {
#pragma unroll
        for (int k = j + 1; k < P; ++k) {
            const double dx = X[k] - X[j], dy = Y[k] - Y[j], dz = Z[k] - Z[j];
            const double d2 = dx * dx + dy * dy + dz * dz;
            const double rh = s.c.hill(j) + s.c.hill(k);
            close |= d2 < rh * rh;
            const double ir3 = 1.0 / (d2 * sqrt(d2));
            ax[j] += s.c.m(k) * dx * ir3;
            ay[j] += s.c.m(k) * dy * ir3;
            az[j] += s.c.m(k) * dz * ir3;
            ax[k] -= s.c.m(j) * dx * ir3;
            ay[k] -= s.c.m(j) * dy * ir3;
            az[k] -= s.c.m(j) * dz * ir3;
        }
    }
    double Ax = a0x, Ay = a0y, Az = a0z;
    bool unbound = false;
#pragma unroll
    for (int i = 0; i < P; ++i) {
        Orbit& o = s.o[i];
        const double jx = ax[i] - Ax, jy = ay[i] - Ay, jz = az[i] - Az;
        const double q = s.c.m(i) / s.c.M(i);
        Ax = Ax + q * jx;
        Ay = Ay + q * jy;
        Az = Az + q * jz;
        const double r2 = o.x * o.x + o.y * o.y + o.z * o.z;
        const double kep = s.c.M(i) / (r2 * sqrt(r2));
        o.vx += h * (jx + kep * o.x);
        o.vy += h * (jy + kep * o.y);
        o.vz += h * (jz + kep * o.z);
        const double alpha = 2.0 / sqrt(r2) - (o.vx * o.vx + o.vy * o.vy + o.vz * o.vz) / s.c.M(i);
        unbound |= !(alpha > 0.0);
    }
    return close || unbound;
}

// Output row k of every trio at time t: each planet's orbit is synchronised on a copy (drift by `half`), so the
// integrated state is untouched.
template <int P>
__device__ __forceinline__ void write_rows(const System<P>& s, double half, const double* __restrict__ el,
                                           double t_over_p1, int k, double* __restrict__ ts_sys) {
#pragma unroll 1
    for (int i = 0; i < P - 2; ++i) {
        double* row = ts_sys + ((int64_t)i * NB_OUT + k) * NB_COLS;
        row[0] = t_over_p1;
#pragma unroll
        for (int c = 1; c < 8; ++c) row[c] = 0.0;
    }
#pragma unroll
    for (int p = 0; p < P; ++p) {
        double e6[6];
        Orbit z = s.o[p];
        if (half != 0.0) kepler_drift(z, s.c.M(p), half);
        orbit_to_elements(z, s.c.M(p), e6);
#pragma unroll
        for (int i = (p > 2 ? p - 2 : 0); i <= (p < P - 3 ? p : P - 3); ++i) {
            double* row = ts_sys + ((int64_t)i * NB_OUT + k) * NB_COLS + 8 + 6 * (p - i);
            row[0] = e6[0] / el[i * 7 + 1];
#pragma unroll
            for (int c = 1; c < 6; ++c) row[c] = e6[c];
        }
    }
}

__device__ __forceinline__ void nan_rows(int n_trios, int k0, double* __restrict__ ts_sys) {
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
#pragma unroll 1
    for (int i = 0; i < n_trios; ++i)
        for (int k = k0; k < NB_OUT; ++k)
            for (int c = 0; c < NB_COLS; ++c) ts_sys[((int64_t)i * NB_OUT + k) * NB_COLS + c] = nan;
}

template <int P>
__global__ void __launch_bounds__(NB_THREADS) nbody_kernel(const double* __restrict__ elements, int64_t n_systems,
                                                           double n_orbits, double dt_frac, double* __restrict__ ts,
                                                           double* __restrict__ masses, double* __restrict__ lt) {
    const int64_t sys = (int64_t)blockIdx.x * NB_THREADS + threadIdx.x;
    if (sys >= n_systems) return;
    const double* el = elements + sys * (P * 7);
    double* ts_sys = ts + sys * ((P - 2) * NB_OUT * NB_COLS);
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
#pragma unroll
    for (int i = 0; i < P - 2; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) masses[(sys * (P - 2) + i) * 3 + j] = el[(i + j) * 7];

    __shared__ double consts[3 * P * NB_THREADS];
    System<P> s;
    s.c.base = consts;
    bool ok = true;
    double acc = 1.0, wmin = 0.0, P1 = 0.0;
#pragma unroll
    for (int i = 0; i < P; ++i) {
        const double m = el[i * 7], a = el[i * 7 + 1], e = el[i * 7 + 2];
        bool fin = true;
#pragma unroll
        for (int c = 0; c < 7; ++c) fin &= isfinite(el[i * 7 + c]);
        ok &= fin && m >= 0.0 && a > 0.0 && e >= 0.0 && e < 1.0;
        acc = acc + m;
        s.c.m(i) = m;
        s.c.M(i) = acc;
        s.c.hill(i) = a * cbrt(m / 3.0);
        const double per = NB_TWO_PI * sqrt(a * a * a / acc);
        const double w = per * ((1.0 - e) * sqrt(1.0 - e) / sqrt(1.0 + e));
        wmin = i == 0 ? w : fmin(wmin, w);
        if (i == 0) P1 = per;
    }
    const double dt = dt_frac * wmin;
    // output k is due at step ceil(t_k / dt); the last one ends the run
    auto out_step = [&](int k) { return ceil((10.0 * k) * n_orbits / 999.0 * P1 / dt); };
    const double last = out_step(NB_OUT - 1);
    if (!ok || !(last <= 2147483648.0)) {
        nan_rows(P - 2, 0, ts_sys);
        lt[sys] = nan;
        return;
    }
    const int64_t n_steps = (int64_t)last;
#pragma unroll
    for (int i = 0; i < P; ++i)
        s.o[i] = elements_to_orbit(s.c.M(i), el[i * 7 + 1], el[i * 7 + 2], el[i * 7 + 3], el[i * 7 + 4], el[i * 7 + 5],
                                   el[i * 7 + 6]);
    int k = 0;
    double next = out_step(0);   // 0
    while (k < NB_OUT && next == 0.0) {
        write_rows<P>(s, 0.0, el, 0.0, k, ts_sys);
        next = ++k < NB_OUT ? out_step(k) : -1.0;
    }
    const double half = 0.5 * dt;
#pragma unroll
    for (int i = 0; i < P; ++i) kepler_drift(s.o[i], s.c.M(i), half);
    for (int64_t step = 1; step <= n_steps; ++step) {
        if (kick<P>(s, dt)) {
            nan_rows(P - 2, k, ts_sys);
            lt[sys] = log10((double)step * dt / P1);
            return;
        }
        if ((double)step == next) {
            const double t_over_p1 = (double)step * dt / P1;
            while (k < NB_OUT && (double)step == next) {
                write_rows<P>(s, half, el, t_over_p1, k, ts_sys);
                next = ++k < NB_OUT ? out_step(k) : -1.0;
            }
        }
        if (step < n_steps) {
#pragma unroll
            for (int i = 0; i < P; ++i) kepler_drift(s.o[i], s.c.M(i), dt);
        }
    }
    lt[sys] = nan;
}

template <int P>
cudaError_t launch(const double* el, int64_t n, double n_orbits, double dt_frac, double* ts, double* ms, double* lt,
                   cudaStream_t st) {
    const int64_t blocks = (n + NB_THREADS - 1) / NB_THREADS;
    nbody_kernel<P><<<(unsigned)blocks, NB_THREADS, 0, st>>>(el, n, n_orbits, dt_frac, ts, ms, lt);
    return cudaGetLastError();
}

}  // namespace
}  // namespace bnn

extern "C" int bnn_integrate_orbits(const double* d_elements, int64_t n_systems, int32_t n_planets, double n_orbits,
                                    double dt_frac, double* d_tseries, double* d_masses, double* d_log10_t_unstable,
                                    void* stream) {
    using namespace bnn;
    // argument checks first: they need no device
    BNN_REQUIRE(d_elements && d_tseries && d_masses && d_log10_t_unstable, BNN_E_ARG, "bnn_integrate_orbits: null pointer");
    BNN_REQUIRE(n_systems >= 1 && n_systems < (1ll << 31), BNN_E_ARG,
                "bnn_integrate_orbits: n_systems = %lld must be in [1, 2^31)", (long long)n_systems);
    BNN_REQUIRE(n_planets >= 3 && n_planets <= 8, BNN_E_ARG, "bnn_integrate_orbits: n_planets = %d must be in [3, 8]",
                (int)n_planets);
    BNN_REQUIRE(isfinite(n_orbits) && n_orbits > 0.0 && isfinite(dt_frac) && dt_frac > 0.0, BNN_E_ARG,
                "bnn_integrate_orbits: n_orbits and dt_frac must be finite and > 0 (got %g, %g)", n_orbits, dt_frac);
    // every system takes at least (990 / 999) n_orbits / dt_frac steps (its dt is at most dt_frac P1)
    BNN_REQUIRE(990.0 * n_orbits / 999.0 / dt_frac <= 2147483648.0, BNN_E_ARG,
                "bnn_integrate_orbits: n_orbits / dt_frac = %g needs more than 2^31 steps", n_orbits / dt_frac);
    const uintptr_t mis = reinterpret_cast<uintptr_t>(d_elements) | reinterpret_cast<uintptr_t>(d_tseries) |
                          reinterpret_cast<uintptr_t>(d_masses) | reinterpret_cast<uintptr_t>(d_log10_t_unstable);
    BNN_REQUIRE((mis & 7u) == 0, BNN_E_ALIGN, "bnn_integrate_orbits: every array must be 8-byte aligned");
    int rc = check_device();
    if (rc != BNN_OK) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaSuccess;
    switch (n_planets) {
        case 3: e = launch<3>(d_elements, n_systems, n_orbits, dt_frac, d_tseries, d_masses, d_log10_t_unstable, st); break;
        case 4: e = launch<4>(d_elements, n_systems, n_orbits, dt_frac, d_tseries, d_masses, d_log10_t_unstable, st); break;
        case 5: e = launch<5>(d_elements, n_systems, n_orbits, dt_frac, d_tseries, d_masses, d_log10_t_unstable, st); break;
        case 6: e = launch<6>(d_elements, n_systems, n_orbits, dt_frac, d_tseries, d_masses, d_log10_t_unstable, st); break;
        case 7: e = launch<7>(d_elements, n_systems, n_orbits, dt_frac, d_tseries, d_masses, d_log10_t_unstable, st); break;
        default: e = launch<8>(d_elements, n_systems, n_orbits, dt_frac, d_tseries, d_masses, d_log10_t_unstable, st); break;
    }
    BNN_CUDA(e);
    return BNN_OK;
}

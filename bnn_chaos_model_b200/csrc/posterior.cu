// K7: posterior post-processing, the step immediately downstream of the predictive kernel (SURVEY 8f rank 1).
//
// Reference (numpy, on the host, over [samples, systems(, trios)] arrays copied back from the GPU):
//   fast_truncnorm(mu, std, left=4, nsamp=40)     figures/main_figures.py:167-223, multiswag_5_planet.py:306-360
//       draw up to nsamp normals x_k = z_k*std + mu, keep the first x_k > left (x_0 if none is)
//   samples >= 9 are re-drawn from the analytic prior on [9, 100]                 main_figures.py:225-259, 5_planet:390-418
//       prior(t) ~ 3.27086190404742 exp(-0.424033970670719 t) - 10.8793430454878 exp(-0.200351029031774 t^2)
//       (the reference inverts a Riemann-sum table of 4*n_samples bins; this file inverts the closed-form CDF)
//   5-planet: min over the adjacent trios of a system, per weight sample            multiswag_5_planet.py:421
//   per system over the weight samples: average, median, percentiles 84 / 16 / 97.5 / 2.5   multiswag_5_planet.py:476-481
//   "median of dists": median of mu and of std over the weight samples              main_figures.py:276-277
//
// Keeping this on the device turns the [N, U, 2] prediction block (48 GB at BASELINE config 3) into [N, 8].
//
// Held-out score of the same block against labels [N, 2]: per system, the log of the ensemble's mean likelihood of the
// label pair and the mean of the per-unit losses, with the model's own loss (VarModel._lossfnc, loss_device.cuh) as the
// per-unit term.  [N, U, 2] -> [N, 2].
//
// Survival probability per system from the same sampled times: the fraction of the U weight samples whose min over trios
// exceeds each of J thresholds, P(T_inst > thr_j), counted exactly.  [N*R, U] -> [N, J].
//
// Variance decomposition of each prediction row of the block: the ensemble's mean mu, the aleatoric part (mean sigma^2),
// and the epistemic part (variance of mu over the units) split into between-model and within-model parts.
// [rows, U, 2] -> [rows, 5].
//
// Which trio sets each system's instability time: per trio row, the fraction of the U weight samples at which that trio
// holds the system's min over trios (first such trio on ties), counted exactly.  [N*R, U] -> [N*R].
//
// The summary, survival and first-trio kernels find a system's trio rows through a row map: UniformRows (every system has R rows,
// system n starts at row n*R) or RaggedRows (a catalogue of mixed planet counts: per-system row offsets in device
// memory, system n owns rows off[n] - off[0] .. off[n+1] - off[0] - 1).  One template per kernel; the uniform entries
// instantiate UniformRows.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "common.cuh"
#include "loss_device.cuh"

namespace bnn {

enum : uint32_t { STREAM_TRUNC = 6, STREAM_PRIOR = 7 };

// prior CDF on [9, inf), un-normalised:  F(t) = A/a (e^{-9a} - e^{-at}) - B sqrt(pi/b)/2 (erf(sqrt(b) t) - erf(9 sqrt(b)))
struct PriorCdf {
    double A = 3.27086190404742, a = 0.424033970670719, B = 10.8793430454878, b = 0.200351029031774;
    __host__ __device__ double cdf(double t) const {
        const double sb = sqrt(b);
        return A / a * (exp(-9.0 * a) - exp(-a * t)) - B * 0.5 * sqrt(3.141592653589793 / b) * (erf(sb * t) - erf(9.0 * sb));
    }
};

// inverse of the normalised prior CDF restricted to [9, 100] (the reference's table ends at top = 100).
// Past t = 12 the Gaussian term of F is the constant K2 = C2 (1 - erf(9 sqrt b)) = 2.6e-7, so F(t) = target has the
// closed-form solution t0 = -log(e^{-9a} - (target + K2) a / A) / a; two Newton steps on the full F take care of
// t < 12 (|t0 - t| <= 4e-6 there).  Equal to a 48-step bisection to < 1e-10 for r <= 1 - 1e-9 (a float32-identical
// result on 40,000 random draws) at 1/14 of its double-precision transcendentals -- the bisection made this
// element-wise kernel 100+ ms at BASELINE config 3 (7.5e8 draws, ~15 % of them resampled, every warp affected).
__device__ __forceinline__ float prior_inverse_cdf(double r) {
    constexpr double A = 3.27086190404742, a = 0.424033970670719, B = 10.8793430454878, b = 0.200351029031774;
    constexpr double E9 = 0.022008957794110346;      // exp(-9 a)
    constexpr double E100 = 3.840949877010102e-19;   // exp(-100 a)
    constexpr double C2 = 21.540303743368245;        // B sqrt(pi / b) / 2
    constexpr double ERF9 = 0.999999987813242;       // erf(9 sqrt(b))
    constexpr double SB = 0.44760588583236255;       // sqrt(b)
    constexpr double TOTAL = 0.16976977144310978;    // F(100)
    const double target = r * TOTAL;
    double arg = E9 - (target + C2 * (1.0 - ERF9)) * (a / A);
    arg = arg > E100 ? arg : E100;
    double t = -log(arg) / a;
#pragma unroll 1
    for (int it = 0; it < 2; ++it) {
        const double e1 = exp(-a * t);
        const double f = A / a * (E9 - e1) - C2 * (erf(SB * t) - ERF9) - target;
        const double fp = A * e1 - B * exp(-b * t * t);
        t -= f / fp;
    }
    t = t < 9.0 ? 9.0 : (t > 100.0 ? 100.0 : t);
    return (float)t;
}

// t[row][u] for every (row = system*R + trio, unit) of pred[rows][U][2]
__global__ void __launch_bounds__(256) sample_instability_kernel(const float2* __restrict__ pred, int64_t total, int64_t U,
                                                                 uint64_t seed, int64_t row_offset, float left, int nsamp,
                                                                 float* __restrict__ t) {
    const int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (idx >= total) return;
    const float2 ms = pred[idx];
    const uint32_t row = (uint32_t)(row_offset + idx / U), u = (uint32_t)(idx % U);  // global row: shard-independent draws
    float first = 0.f, val = 0.f;
    bool found = false;
    for (int k4 = 0; k4 * 4 < nsamp && !found; ++k4) {
        const float4 z = philox_normal4_fast(seed, STREAM_TRUNC, u, row, (uint32_t)k4);  // special-function-unit Box-Muller (1e-6 abs)
        const float zz[4] = {z.x, z.y, z.z, z.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            if (found || 4 * k4 + i >= nsamp) break;
            const float x = __fadd_rn(__fmul_rn(zz[i], ms.y), ms.x);  // rand_out * scale + loc
            if (k4 == 0 && i == 0) first = x;
            if (x > left) { val = x; found = true; }
        }
    }
    if (!found) val = first;  // mask.argmax(0) == 0 when no draw passes
    if (val >= 9.0f) {        // stable_past_9: resample from the prior
        const uint4 rr = philox4x32_10(make_uint4(0u, u, row, STREAM_PRIOR), make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
        const double r = ((double)rr.x * 4294967296.0 + (double)rr.y) * (1.0 / 18446744073709551616.0);  // [0,1)
        val = prior_inverse_cdf(r);
    }
    t[idx] = val;
}

// ---- which rows belong to system n (rows are system-major: a system's trio rows are contiguous) ----
struct UniformRows {   // every system has R trio rows; the first one, n*R, is formed where it is used
    int R;
    struct Span {
        int64_t n;
        int R;
        __device__ __forceinline__ int64_t first() const { return n * R; }
        __device__ __forceinline__ int count() const { return R; }
    };
    __device__ __forceinline__ Span operator()(int64_t n) const { return {n, R}; }
    static __device__ __forceinline__ bool empty(const Span&) { return false; }
};
struct RaggedRows {    // per-system counts as offsets [n_systems + 1]; rows are counted from off[0]
    const int64_t* __restrict__ off;
    struct Span {
        int64_t first_, count_;
        __device__ __forceinline__ int64_t first() const { return first_; }
        __device__ __forceinline__ int64_t count() const { return count_; }
    };
    __device__ __forceinline__ Span operator()(int64_t n) const {   // read once per CTA
        const int64_t o0 = off[0], a = off[n], b = off[n + 1];
        return {a - o0, b - a};
    }
    // a count <= 0 (malformed offsets) gives a NaN row instead of a read outside the block
    static __device__ __forceinline__ bool empty(const Span& s) { return s.count_ <= 0; }
};

// ---- per-system order statistics over the weight samples: bitonic sort in shared memory ----
__device__ __forceinline__ void bitonic_sort(float* s, int n) {
    for (int k = 2; k <= n; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < n; i += blockDim.x) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const float a = s[i], b = s[ixj];
                    const bool up = (i & k) == 0;
                    if ((a > b) == up) { s[i] = b; s[ixj] = a; }
                }
            }
            __syncthreads();
        }
    }
}

// numpy.percentile(method='linear'): virtual index q/100 (n-1), lerp with numpy's t >= 0.5 fix-up
__device__ __forceinline__ float percentile_sorted(const float* s, int n, double q) {
    const double pos = q / 100.0 * (double)(n - 1);
    int lo = (int)floor(pos);
    lo = max(0, min(lo, n - 1));
    const int hi = min(lo + 1, n - 1);
    const double tfrac = pos - (double)lo;
    const double a = s[lo], b = s[hi];
    const double d = b - a;
    return (float)(tfrac >= 0.5 ? b - d * (1.0 - tfrac) : a + d * tfrac);
}

__device__ __forceinline__ float block_sum(float v, float* red) {
    __syncthreads();
    red[threadIdx.x] = v;
    __syncthreads();
    for (int st = blockDim.x >> 1; st > 0; st >>= 1) {
        if ((int)threadIdx.x < st) red[threadIdx.x] += red[threadIdx.x + st];
        __syncthreads();
    }
    return red[0];
}

// one CTA per system.  t[(first + r)*U + u]; pred[(first + r)*U + u] = (mu, std), r < count (the system's Rows span).  stats[n][8]:
// average, median, p84, p16, p97.5, p2.5 of min_r t; median over units of mu* = min_r mu and of its std.
template <class Rows>
__global__ void __launch_bounds__(512) summarize_instability_kernel(const float* __restrict__ t, const float2* __restrict__ pred,
                                                                    Rows rows, int U, int n_pow2, float* __restrict__ stats) {
    extern __shared__ float sh[];
    float* s = sh;               // n_pow2 sort buffer
    float* red = sh + n_pow2;    // blockDim.x
    const int64_t n = blockIdx.x;
    const float INF = __int_as_float(0x7f800000);
    float* out = stats + n * 8;
    const auto sp = rows(n);
    if (Rows::empty(sp)) {   // uniform in the CTA: nobody reaches a barrier
        if (threadIdx.x < 8) out[threadIdx.x] = __int_as_float(0x7fffffff);
        return;
    }
    // ---- min over trios of the sampled time ----
    float part = 0.f;
    for (int u = threadIdx.x; u < n_pow2; u += blockDim.x) {
        float v = INF;
        if (u < U) {
            for (decltype(sp.count()) r = 0; r < sp.count(); ++r) v = fminf(v, t[(sp.first() + r) * (int64_t)U + u]);
            part += v;
        }
        s[u] = v;
    }
    const float total = block_sum(part, red);
    bitonic_sort(s, n_pow2);
    if (threadIdx.x == 0) {
        out[0] = total / (float)U;
        out[1] = percentile_sorted(s, U, 50.0);
        out[2] = percentile_sorted(s, U, 50.0 + 68.0 / 2);
        out[3] = percentile_sorted(s, U, 50.0 - 68.0 / 2);
        out[4] = percentile_sorted(s, U, 50.0 + 95.0 / 2);
        out[5] = percentile_sorted(s, U, 50.0 - 95.0 / 2);
    }
    __syncthreads();
    // ---- median of dists: mu* = min over trios of mu, std* = std of that trio ----
    for (int pass = 0; pass < 2; ++pass) {
        for (int u = threadIdx.x; u < n_pow2; u += blockDim.x) {
            float v = INF;
            if (u < U) {
                float best = INF, bsd = 0.f;
                for (decltype(sp.count()) r = 0; r < sp.count(); ++r) {
                    const float2 p = pred[(sp.first() + r) * (int64_t)U + u];
                    if (p.x < best || r == 0) { best = p.x; bsd = p.y; }
                }
                v = pass == 0 ? best : bsd;
                if (!(v == v)) v = INF;  // NaN predictions sort last
            }
            s[u] = v;
        }
        __syncthreads();
        bitonic_sort(s, n_pow2);
        if (threadIdx.x == 0) out[6 + pass] = percentile_sorted(s, U, 50.0);
        __syncthreads();
    }
}

// ---- the same statistics for any U: exact order statistics by 3-pass radix select (11 + 11 + 10 bits of an
// order-preserving key) with shared-memory histograms, one per requested rank; nothing is sorted or stored ----
constexpr int SEL_MAXT = 10;  // ranks per array: floor / ceil neighbours of 5 percentiles

__device__ __forceinline__ uint32_t order_key(float v) {
    if (!(v == v)) v = __int_as_float(0x7f800000);  // NaN predictions rank last, like the sort path
    const uint32_t b = __float_as_uint(v);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float key_value(uint32_t k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

// which: 0 = min over trios of t, 1 = mu* (min over trios of mu), 2 = std of the arg-min trio, over the rows of sp
template <class Span>
__device__ __forceinline__ float summary_value(const float* __restrict__ t, const float2* __restrict__ pred, const Span& sp,
                                               int U, int u, int which) {
    if (which == 0) {
        float v = __int_as_float(0x7f800000);
        for (decltype(sp.count()) r = 0; r < sp.count(); ++r) v = fminf(v, t[(sp.first() + r) * (int64_t)U + u]);
        return v;
    }
    float best = 0.f, bsd = 0.f;
    for (decltype(sp.count()) r = 0; r < sp.count(); ++r) {
        const float2 p = pred[(sp.first() + r) * (int64_t)U + u];
        if (r == 0 || p.x < best) { best = p.x; bsd = p.y; }
    }
    return which == 1 ? best : bsd;
}

// histogram increment with the lanes of a warp that hit the same bin merged into one shared-memory atomic: the sampled
// times of a system sit in a handful of top-11-bit bins (sign + exponent + 2 mantissa bits), where plain atomics serialise
__device__ __forceinline__ void hist_add_warp(uint32_t* __restrict__ hist, uint32_t bin, bool valid) {
    const uint32_t act = __ballot_sync(0xffffffffu, valid);
    if (valid) {
        const uint32_t peers = __match_any_sync(act, bin);
        if ((threadIdx.x & 31) == (uint32_t)(__ffs(peers) - 1)) atomicAdd(&hist[bin], (uint32_t)__popc(peers));
    }
}

// warp `w` finds the bin holding rank[w] in hist (nbins <= 2048 counts): returns the bin, updates the rank to the
// rank inside the bin
__device__ __forceinline__ int select_bin(const uint32_t* __restrict__ hist, int nbins, uint32_t& rank) {
    const int lane = threadIdx.x & 31;
    const int per = nbins / 32;
    uint32_t mine = 0;
    for (int i = 0; i < per; ++i) mine += hist[lane * per + i];
    uint32_t incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t up = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += up;
    }
    const uint32_t excl = incl - mine;
    const uint32_t ballot = __ballot_sync(0xffffffffu, rank < incl);
    const int src = __ffs(ballot) - 1;  // first lane whose inclusive count exceeds the rank
    int bin = 0;
    uint32_t r = 0;
    if (lane == src) {
        r = rank - excl;
        for (int i = 0; i < per; ++i) {
            const uint32_t c = hist[lane * per + i];
            if (r < c) { bin = lane * per + i; break; }
            r -= c;
        }
    }
    bin = __shfl_sync(0xffffffffu, bin, src);
    rank = __shfl_sync(0xffffffffu, r, src);
    return bin;
}

template <class Rows>
__global__ void __launch_bounds__(512) summarize_select_kernel(const float* __restrict__ t, const float2* __restrict__ pred,
                                                               Rows rows, int U, float* __restrict__ stats) {
    extern __shared__ uint32_t hist[];            // [SEL_MAXT][2048]
    __shared__ uint32_t s_rank[SEL_MAXT], s_prefix[SEL_MAXT];
    __shared__ float s_val[SEL_MAXT], red[512];
    const int64_t n = blockIdx.x;
    const int warp = threadIdx.x >> 5;
    float* out = stats + n * 8;
    const auto sp = rows(n);
    if (Rows::empty(sp)) {   // uniform in the CTA: nobody reaches a barrier
        if (threadIdx.x < 8) out[threadIdx.x] = __int_as_float(0x7fffffff);
        return;
    }
    const double qs[5] = {50.0, 50.0 + 68.0 / 2, 50.0 - 68.0 / 2, 50.0 + 95.0 / 2, 50.0 - 95.0 / 2};
    for (int which = 0; which < 3; ++which) {
        const int nq = which == 0 ? 5 : 1, nt = 2 * nq;
        if (threadIdx.x < nt) {
            const double pos = qs[threadIdx.x >> 1] / 100.0 * (double)(U - 1);
            int lo = (int)floor(pos);
            lo = max(0, min(lo, U - 1));
            s_rank[threadIdx.x] = (threadIdx.x & 1) ? min(lo + 1, U - 1) : lo;
            s_prefix[threadIdx.x] = 0;
        }
        // pass 1: top 11 bits, one histogram for every target (+ the sum for the average)
        for (int i = threadIdx.x; i < 2048; i += blockDim.x) hist[i] = 0;
        __syncthreads();
        float part = 0.f;
        for (int u0 = 0; u0 < U; u0 += blockDim.x) {   // whole warps stay in the loop: the merge below is warp-collective
            const int u = u0 + threadIdx.x;
            const bool valid = u < U;
            const float v = valid ? summary_value(t, pred, sp, U, u, which) : 0.f;
            if (valid) part += v;
            hist_add_warp(hist, order_key(v) >> 21, valid);
        }
        if (which == 0) {
            const float total = block_sum(part, red);
            if (threadIdx.x == 0) out[0] = total / (float)U;
        }
        __syncthreads();
        if (warp < nt) {
            uint32_t r = s_rank[warp];
            const int b = select_bin(hist, 2048, r);
            if ((threadIdx.x & 31) == 0) { s_rank[warp] = r; s_prefix[warp] = (uint32_t)b; }
        }
        __syncthreads();
        // pass 2: next 11 bits, pass 3: last 10 bits -- one histogram per target, restricted to its prefix
        for (int pass = 0; pass < 2; ++pass) {
            const int bits = pass == 0 ? 11 : 10, shift = pass == 0 ? 10 : 0, nb = 1 << bits;
            for (int i = threadIdx.x; i < nt * 2048; i += blockDim.x) hist[i] = 0;
            __syncthreads();
            for (int u = threadIdx.x; u < U; u += blockDim.x) {
                const uint32_t k = order_key(summary_value(t, pred, sp, U, u, which));
                const uint32_t pre = k >> (shift + bits);
                for (int tt = 0; tt < nt; ++tt)
                    if (pre == s_prefix[tt]) atomicAdd(&hist[tt * 2048 + ((k >> shift) & (nb - 1))], 1u);
            }
            __syncthreads();
            if (warp < nt) {
                uint32_t r = s_rank[warp];
                const int b = select_bin(hist + warp * 2048, nb, r);
                if ((threadIdx.x & 31) == 0) { s_rank[warp] = r; s_prefix[warp] = (s_prefix[warp] << bits) | (uint32_t)b; }
            }
            __syncthreads();
        }
        if (threadIdx.x < nt) s_val[threadIdx.x] = key_value(s_prefix[threadIdx.x]);
        __syncthreads();
        if (threadIdx.x < nq) {
            const double pos = qs[threadIdx.x] / 100.0 * (double)(U - 1);
            int lo = (int)floor(pos);
            lo = max(0, min(lo, U - 1));
            const double tfrac = pos - (double)lo;
            const double a = s_val[2 * threadIdx.x], b = s_val[2 * threadIdx.x + 1], d = b - a;
            const float v = (float)(tfrac >= 0.5 ? b - d * (1.0 - tfrac) : a + d * tfrac);  // numpy's lerp
            if (which == 0) out[1 + threadIdx.x] = v; else out[5 + which] = v;
        }
        __syncthreads();
    }
}

// ---- held-out score: one CTA per system.  loss[u] = -(l(y0) + l(y1)) of nll_terms, bit for bit bnn_nll_fwd_bwd's
// per-system loss.  Each thread walks the units tid, tid + 256, ... keeping, in double, m = max of -loss, s = sum of
// exp(-loss - m) (rescaled when m grows) and t = sum of loss; the 256 partials are merged by a fixed tree.  No atomics:
// a row's result is a function of that row's inputs alone, and repeated calls are bit-identical.
constexpr int SCORE_THREADS = 256;

// (m, s) <- (m, s) merged with (m2, s2); s == 0 marks a partial that has seen no finite term
__device__ __forceinline__ void lse_merge(double& m, double& s, double m2, double s2) {
    if (s2 == 0.0) return;
    if (s == 0.0) { m = m2; s = s2; return; }
    if (m2 > m) { s = s * exp(m - m2) + s2; m = m2; }
    else s += s2 * exp(m2 - m);
}

__global__ void __launch_bounds__(SCORE_THREADS) score_labels_kernel(const float2* __restrict__ pred, int64_t U,
                                                                     const float2* __restrict__ y, float2* __restrict__ score) {
    __shared__ double sh_m[SCORE_THREADS], sh_s[SCORE_THREADS], sh_t[SCORE_THREADS];
    const int64_t n = blockIdx.x;
    const int tid = threadIdx.x;
    const float2 yy = y[n];
    const float2* __restrict__ p = pred + n * U;
    const double NEG_INF = -__longlong_as_double(0x7ff0000000000000ll);
    double m = NEG_INF, s = 0.0, t = 0.0;
    for (int64_t u = tid; u < U; u += SCORE_THREADS) {
        const float2 ms = p[u];
        float l0, l1, d0, d1;
        nll_terms(ms.x, ms.y, yy.x, l0, d0, d1);
        nll_terms(ms.x, ms.y, yy.y, l1, d0, d1);
        const float loss = -(l0 + l1);
        const double v = -(double)loss;
        t += (double)loss;
        if (v > m) { s = s * exp(m - v) + 1.0; m = v; }
        else if (v > NEG_INF) s += exp(v - m);   // -inf only when l0 + l1 overflows fp32: it adds nothing
    }
    sh_m[tid] = m; sh_s[tid] = s; sh_t[tid] = t;
    __syncthreads();
    for (int w = SCORE_THREADS / 2; w > 0; w >>= 1) {
        if (tid < w) {
            lse_merge(m, s, sh_m[tid + w], sh_s[tid + w]);
            t += sh_t[tid + w];
            sh_m[tid] = m; sh_s[tid] = s; sh_t[tid] = t;
        }
        __syncthreads();
    }
    if (tid == 0) {
        const double lpd = m + (log(s) - log((double)U));   // log((1/U) sum_u exp(-loss[u]))
        score[n] = make_float2((float)lpd, (float)(t / (double)U));
    }
}

// ---- survival: one CTA per system.  tmin[u] = min over trios of t, fminf from +inf exactly as the summary computes it
// (a unit whose trio draws are all NaN counts as +inf); bin(u) = number of thresholds strictly below tmin[u], found by a
// binary search over the ascending thresholds and counted in per-warp shared-memory histograms; then
// count_j = #{u : bin(u) > j}, a suffix sum.  Integer counts: a row's result depends on that row alone and repeated
// calls are bit-identical.
constexpr int SURV_THREADS = 256, SURV_MAXJ = 64, SURV_UNROLL = 4;

struct SurvivalThresholds {   // passed by value in the kernel's parameters
    float thr[SURV_MAXJ];      // ascending
    int32_t col[SURV_MAXJ];    // output column of thr[j]
    int32_t J;
};

template <class Rows>
__global__ void __launch_bounds__(SURV_THREADS) survival_kernel(const float* __restrict__ t, Rows sys_rows, int64_t U,
                                                                const __grid_constant__ SurvivalThresholds th,
                                                                float* __restrict__ surv) {
    constexpr int WARPS = SURV_THREADS / 32;
    __shared__ float s_thr[SURV_MAXJ];
    __shared__ uint32_t hist[WARPS][SURV_MAXJ + 1], s_tot[SURV_MAXJ + 1];
    const int tid = threadIdx.x, J = th.J;
    const float INF = __int_as_float(0x7f800000);
    const int64_t n = blockIdx.x;
    const auto sp = sys_rows(n);
    if (Rows::empty(sp)) {   // uniform in the CTA: nobody reaches a barrier
        if (tid < J) surv[n * J + tid] = __int_as_float(0x7fffffff);
        return;
    }
    if (tid < J) s_thr[tid] = th.thr[tid];
    for (int i = tid; i < WARPS * (SURV_MAXJ + 1); i += SURV_THREADS) (&hist[0][0])[i] = 0;
    __syncthreads();
    const float* __restrict__ rows = t + sp.first() * U;
    uint32_t* __restrict__ h = hist[tid >> 5];
    // whole warps stay in the loop: hist_add_warp is warp-collective
    for (int64_t u0 = 0; u0 < U; u0 += SURV_THREADS * SURV_UNROLL) {
        float v[SURV_UNROLL];
#pragma unroll
        for (int k = 0; k < SURV_UNROLL; ++k) v[k] = INF;
        for (decltype(sp.count()) r = 0; r < sp.count(); ++r) {   // SURV_UNROLL independent coalesced loads in flight per trio row
#pragma unroll
            for (int k = 0; k < SURV_UNROLL; ++k) {
                const int64_t u = u0 + k * SURV_THREADS + tid;
                if (u < U) v[k] = fminf(v[k], rows[r * U + u]);
            }
        }
#pragma unroll
        for (int k = 0; k < SURV_UNROLL; ++k) {
            int b = 0;   // #{j : thr[j] < v}: the predicate is monotone in j, so the greedy power-of-two steps find it
#pragma unroll
            for (int step = SURV_MAXJ; step > 0; step >>= 1)
                if (b + step <= J && s_thr[b + step - 1] < v[k]) b += step;
            hist_add_warp(h, (uint32_t)b, u0 + k * SURV_THREADS + tid < U);
        }
    }
    __syncthreads();
    if (tid <= J) {
        uint32_t c = 0;
        for (int w = 0; w < WARPS; ++w) c += hist[w][tid];
        s_tot[tid] = c;
    }
    __syncthreads();
    if (tid < J) {
        uint32_t c = 0;   // tmin > thr[tid]  <=>  bin > tid
        for (int b = tid + 1; b <= J; ++b) c += s_tot[b];
        surv[n * J + th.col[tid]] = (float)((double)c / (double)U);
    }
}

// ---- which trio sets the system's min: one CTA per system.  tmin[u] = fminf over the system's rows from +inf, as the
// summary takes it; the winner of unit u is the first row r with t[r][u] == tmin[u], found as a running (best, index)
// pair that a row takes over when it is strictly smaller, or when it is the first non-NaN row (so a +inf row can win).
// A unit whose draws are all NaN has no winner.  Per-trio winner counts in one CTA-wide shared-memory histogram; integer
// counts: a system's result depends on its own rows only and repeated calls are bit-identical.
constexpr int FIRST_THREADS = 256, FIRST_UNROLL = 4, FIRST_MAXR = 1024;

template <class Rows>
__global__ void __launch_bounds__(FIRST_THREADS) first_trio_kernel(const float* __restrict__ t, Rows sys_rows, int64_t U,
                                                                   float* __restrict__ first) {
    __shared__ uint32_t hist[FIRST_MAXR];
    const int tid = threadIdx.x;
    const float INF = __int_as_float(0x7f800000);
    const auto sp = sys_rows(blockIdx.x);
    if (sp.count() <= 0) return;   // owns no rows: nothing to write (uniform in the CTA: nobody reaches a barrier)
    float* __restrict__ out = first + sp.first();
    if (sp.count() > FIRST_MAXR) {   // more trios than counters (ragged only: the uniform entry refuses it)
        for (int64_t r = tid; r < sp.count(); r += FIRST_THREADS) out[r] = __int_as_float(0x7fffffff);
        return;
    }
    const int R = (int)sp.count();
    for (int i = tid; i < R; i += FIRST_THREADS) hist[i] = 0;
    __syncthreads();
    const float* __restrict__ rows = t + sp.first() * U;
    // whole warps stay in the loop: hist_add_warp is warp-collective
    for (int64_t u0 = 0; u0 < U; u0 += FIRST_THREADS * FIRST_UNROLL) {
        float best[FIRST_UNROLL];
        int idx[FIRST_UNROLL];
#pragma unroll
        for (int k = 0; k < FIRST_UNROLL; ++k) { best[k] = INF; idx[k] = -1; }
        for (int r = 0; r < R; ++r) {   // FIRST_UNROLL independent coalesced loads in flight per trio row
#pragma unroll
            for (int k = 0; k < FIRST_UNROLL; ++k) {
                const int64_t u = u0 + k * FIRST_THREADS + tid;
                if (u < U) {
                    const float v = rows[r * U + u];
                    if (v < best[k] || (idx[k] < 0 && v == v)) { best[k] = v; idx[k] = r; }
                }
            }
        }
#pragma unroll
        for (int k = 0; k < FIRST_UNROLL; ++k)
            hist_add_warp(hist, (uint32_t)idx[k], u0 + k * FIRST_THREADS + tid < U && idx[k] >= 0);
    }
    __syncthreads();
    for (int r = tid; r < R; r += FIRST_THREADS) out[r] = (float)((double)hist[r] / (double)U);
}

// ---- variance decomposition: one CTA per prediction row, unit u = k*S + s of model k.  Pass 1: the units of a warp's
// 32 lanes are consecutive, so their model indices are sorted and form a few contiguous segments; a segmented shuffle
// scan sums each segment and its last lane adds the sum to the warp's own accumulator acc[warp][k] in shared memory.
// The model sums are then the sums over warps in warp order.  Pass 2 re-reads the row for (mu - m_k)^2 against the model
// means.  Everything accumulates in double in a fixed order with no atomics: a row's result depends on that row alone.
constexpr int UNC_THREADS = 256, UNC_WARPS = UNC_THREADS / 32, UNC_UNROLL = 4, UNC_MAXM = 1024;

// sum over the CTA, the same bits in every thread: xor butterfly (commutative pairs, so every lane agrees) + warp order
__device__ __forceinline__ double block_sum_d(double v, double* red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();   // red may still be read by the previous call
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < UNC_WARPS; ++w) s += red[w];
    return s;
}

__global__ void __launch_bounds__(UNC_THREADS) uncertainty_kernel(const float2* __restrict__ pred, int64_t U, uint32_t S,
                                                                  int M, float* __restrict__ out) {
    extern __shared__ double acc[];   // [UNC_WARPS][M] per-warp model sums of mu; then acc[k] = m_k
    __shared__ double red[UNC_WARPS];
    const int tid = threadIdx.x, lane = tid & 31;
    const int64_t row = blockIdx.x;
    const float2* __restrict__ p = pred + row * U;
    for (int i = tid; i < UNC_WARPS * M; i += UNC_THREADS) acc[i] = 0.0;
    __syncthreads();
    double* __restrict__ mine = acc + (tid >> 5) * M;
    double sd2 = 0.0;
    bool bad_mu = false, bad_sd = false;
    // pass 1: model sums of mu, sum of sigma^2.  Whole warps stay in the loop: the scan is warp-collective.
    for (int64_t u0 = 0; u0 < U; u0 += UNC_THREADS * UNC_UNROLL) {
        float2 v[UNC_UNROLL];
#pragma unroll
        for (int k = 0; k < UNC_UNROLL; ++k) {   // UNC_UNROLL independent coalesced loads in flight
            const int64_t u = u0 + k * UNC_THREADS + tid;
            v[k] = u < U ? p[u] : make_float2(0.f, 0.f);
        }
#pragma unroll
        for (int k = 0; k < UNC_UNROLL; ++k) {
            const int64_t u = u0 + k * UNC_THREADS + tid;
            const bool valid = u < U;
            bad_mu |= !isfinite(v[k].x);
            bad_sd |= !isfinite(v[k].y);
            sd2 += (double)v[k].y * (double)v[k].y;
            const uint32_t model = valid ? (uint32_t)u / S : (uint32_t)M;
            const uint32_t peers = __match_any_sync(0xffffffffu, model);
            const int first = __ffs(peers) - 1;
            double s = (double)v[k].x;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const double up = __shfl_up_sync(0xffffffffu, s, d);
                if (lane - d >= first) s += up;
            }
            if (valid && lane == 31 - __clz(peers)) mine[model] += s;
            __syncwarp();   // the next segment's lane may update the same entry
        }
    }
    __syncthreads();
    // model means m_k, their mean, and the between-model moment
    double part = 0.0;
    for (int k = tid; k < M; k += UNC_THREADS) {
        double s = 0.0;
        for (int w = 0; w < UNC_WARPS; ++w) s += acc[w * M + k];
        const double m = s / (double)S;
        acc[k] = m;   // column k is read by this thread only
        part += m;
    }
    const double mean = block_sum_d(part, red) / (double)M;   // its barriers publish acc[k]
    part = 0.0;
    for (int k = tid; k < M; k += UNC_THREADS) {
        const double d = acc[k] - mean;
        part += d * d;
    }
    const double between = block_sum_d(part, red) / (double)M;
    // pass 2: within-model moment (1/M) sum_k (1/S) sum_s (mu - m_k)^2 = (1/U) sum_u (mu_u - m_k(u))^2
    part = 0.0;
    for (int64_t u0 = 0; u0 < U; u0 += UNC_THREADS * UNC_UNROLL) {
        float mu[UNC_UNROLL];
#pragma unroll
        for (int k = 0; k < UNC_UNROLL; ++k) {
            const int64_t u = u0 + k * UNC_THREADS + tid;
            mu[k] = u < U ? p[u].x : 0.f;
        }
#pragma unroll
        for (int k = 0; k < UNC_UNROLL; ++k) {
            const int64_t u = u0 + k * UNC_THREADS + tid;
            if (u < U) {
                const double d = (double)mu[k] - acc[(uint32_t)u / S];
                part += d * d;
            }
        }
    }
    const double within = block_sum_d(part, red) / (double)U;
    const double aleatoric = block_sum_d(sd2, red) / (double)U;
    const int nonfinite_mu = __syncthreads_or(bad_mu), nonfinite_sd = __syncthreads_or(bad_sd);
    if (tid == 0) {
        const float NaN = __int_as_float(0x7fffffff);
        float* o = out + row * 5;
        o[0] = nonfinite_mu ? NaN : (float)mean;
        o[1] = nonfinite_sd ? NaN : (float)aleatoric;
        o[2] = nonfinite_mu ? NaN : (float)(between + within);
        o[3] = nonfinite_mu ? NaN : (float)between;
        o[4] = nonfinite_mu ? NaN : (float)within;
    }
}

}  // namespace bnn

extern "C" {

int bnn_sample_instability(const float* d_pred, int64_t n_rows, int64_t n_units, uint64_t seed, int64_t row_offset,
                           float left, int32_t nsamp, float* d_t, void* stream) {
    using namespace bnn;
    int rc = check_device();
    if (rc != BNN_OK) return rc;
    BNN_REQUIRE(d_pred && d_t && n_rows > 0 && n_units > 0 && nsamp >= 1, BNN_E_ARG,
                "bnn_sample_instability: null pointer or empty problem");
    BNN_REQUIRE(row_offset >= 0 && row_offset + n_rows < (1ll << 32) && n_units < (1ll << 32), BNN_E_ARG,
                "bnn_sample_instability: index exceeds 32 bits");
    const int64_t total = n_rows * n_units;
    const int64_t blocks = (total + 255) / 256;
    BNN_REQUIRE(blocks < (1ll << 31), BNN_E_ARG, "bnn_sample_instability: too many elements for one launch");
    sample_instability_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>((const float2*)d_pred, total, n_units, seed,
                                                                                 row_offset, left, nsamp, d_t);
    BNN_CUDA(cudaGetLastError());
    return BNN_OK;
}

// 0 = automatic (shared-memory sort while it fits, else radix select), 1 = radix select; process-wide diagnostic override
// (bnn_set_summary_variant), default read once from BNN_SUMMARY_VARIANT = select
static int g_summary_variant = -1;
static int summary_variant() {
    if (g_summary_variant < 0) {
        const char* force = getenv("BNN_SUMMARY_VARIANT");
        g_summary_variant = (force && !strcmp(force, "select")) ? 1 : 0;
    }
    return g_summary_variant;
}
int bnn_set_summary_variant(int32_t variant) {
    BNN_REQUIRE(variant == 0 || variant == 1, BNN_E_ARG, "bnn_set_summary_variant: 0 = auto, 1 = radix select");
    g_summary_variant = variant;
    return BNN_OK;
}

}  // extern "C"

namespace {

// summary launch for either row map: the shared-memory sort while U fits, else (or when forced) the radix select
template <class Rows>
int launch_summary(const float* d_t, const float* d_pred, int64_t n_systems, Rows rows, int32_t n_units, float* d_stats,
                   void* stream) {
    using namespace bnn;
    int n_pow2 = 1;
    while (n_pow2 < n_units) n_pow2 <<= 1;
    const int threads = 512;
    const size_t smem = (size_t)(n_pow2 + threads) * sizeof(float);
    const bool use_select = summary_variant() == 1 || smem > 200 * 1024;   // 1: forced (tests cross-check the two)
    if (use_select) {
        // more weight samples than the shared-memory sort holds (30 models x 2000 samples = 60000 at BASELINE config 3):
        // exact order statistics by radix select, nothing is stored
        const size_t hsm = (size_t)SEL_MAXT * 2048 * sizeof(uint32_t);
        static PerDeviceOnce attr2_done;
        if (attr2_done.need()) {
            BNN_CUDA(cudaFuncSetAttribute(summarize_select_kernel<Rows>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          200 * 1024));
        }
        summarize_select_kernel<Rows><<<(unsigned)n_systems, threads, hsm, (cudaStream_t)stream>>>(
            d_t, (const float2*)d_pred, rows, n_units, d_stats);
        BNN_CUDA(cudaGetLastError());
        return BNN_OK;
    }
    static PerDeviceOnce attr_done;
    if (attr_done.need()) {
        BNN_CUDA(cudaFuncSetAttribute(summarize_instability_kernel<Rows>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      200 * 1024));
    }
    summarize_instability_kernel<Rows><<<(unsigned)n_systems, threads, smem, (cudaStream_t)stream>>>(
        d_t, (const float2*)d_pred, rows, n_units, n_pow2, d_stats);
    BNN_CUDA(cudaGetLastError());
    return BNN_OK;
}

// the thresholds sorted ascending, with their output columns, for the kernel's parameters; BNN_E_ARG on a NaN
int survival_thresholds(const char* what, const float* h_thresholds, int32_t n_thresholds, bnn::SurvivalThresholds& th) {
    using namespace bnn;
    BNN_REQUIRE(n_thresholds >= 1 && n_thresholds <= SURV_MAXJ, BNN_E_ARG,
                "%s: n_thresholds must be in [1, %d], got %d", what, SURV_MAXJ, (int)n_thresholds);
    for (int j = 0; j < n_thresholds; ++j)
        BNN_REQUIRE(!isnan(h_thresholds[j]), BNN_E_ARG, "%s: threshold %d is NaN", what, j);
    th.J = n_thresholds;
    for (int j = 0; j < n_thresholds; ++j) th.col[j] = j;
    std::stable_sort(th.col, th.col + n_thresholds, [&](int a, int b) { return h_thresholds[a] < h_thresholds[b]; });
    for (int j = 0; j < n_thresholds; ++j) th.thr[j] = h_thresholds[th.col[j]];
    for (int j = n_thresholds; j < SURV_MAXJ; ++j) { th.thr[j] = 0.f; th.col[j] = 0; }
    return BNN_OK;
}

bool aligned(const void* q, uintptr_t bytes) { return (reinterpret_cast<uintptr_t>(q) & (bytes - 1)) == 0; }

}  // namespace

extern "C" {

int bnn_summarize_instability(const float* d_t, const float* d_pred, int64_t n_systems, int32_t n_trios, int32_t n_units,
                              float* d_stats, void* stream) {
    using namespace bnn;
    int rc = check_device();
    if (rc != BNN_OK) return rc;
    BNN_REQUIRE(d_t && d_pred && d_stats && n_systems > 0 && n_trios > 0 && n_units > 0, BNN_E_ARG,
                "bnn_summarize_instability: null pointer or empty problem");
    BNN_REQUIRE(n_systems < (1ll << 31), BNN_E_ARG, "bnn_summarize_instability: too many systems for one launch");
    return launch_summary(d_t, d_pred, n_systems, UniformRows{n_trios}, n_units, d_stats, stream);
}

int bnn_summarize_instability_ragged(const float* d_t, const float* d_pred, int64_t n_systems,
                                     const int64_t* d_row_offsets, int32_t n_units, float* d_stats, void* stream) {
    using namespace bnn;
    // argument checks first: they need no device
    BNN_REQUIRE(d_t && d_pred && d_stats && d_row_offsets && n_systems > 0 && n_units > 0, BNN_E_ARG,
                "bnn_summarize_instability_ragged: null pointer or empty problem");
    BNN_REQUIRE(n_systems < (1ll << 31), BNN_E_ARG, "bnn_summarize_instability_ragged: too many systems for one launch");
    BNN_REQUIRE(aligned(d_row_offsets, 8), BNN_E_ALIGN, "bnn_summarize_instability_ragged: d_row_offsets must be 8-byte aligned");
    int rc = check_device();
    if (rc != BNN_OK) return rc;
    return launch_summary(d_t, d_pred, n_systems, RaggedRows{d_row_offsets}, n_units, d_stats, stream);
}

int bnn_score_labels(const float* d_pred, int64_t n_systems, int64_t n_units, const float* d_y, float* d_score,
                     void* stream) {
    using namespace bnn;
    // argument checks first: they need no device
    BNN_REQUIRE(d_pred && d_y && d_score && n_systems > 0 && n_units > 0, BNN_E_ARG,
                "bnn_score_labels: null pointer or empty problem");
    BNN_REQUIRE(n_systems < (1ll << 31) && n_units < (1ll << 32), BNN_E_ARG,
                "bnn_score_labels: n_systems must be < 2^31 and n_units < 2^32");
    const auto aligned8 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 7u) == 0; };
    BNN_REQUIRE(aligned8(d_pred) && aligned8(d_y) && aligned8(d_score), BNN_E_ALIGN,
                "bnn_score_labels: pointers must be 8-byte aligned");
    int rc = check_device();
    if (rc != BNN_OK) return rc;
    score_labels_kernel<<<(unsigned)n_systems, SCORE_THREADS, 0, (cudaStream_t)stream>>>(
        (const float2*)d_pred, n_units, (const float2*)d_y, (float2*)d_score);
    BNN_CUDA(cudaGetLastError());
    return BNN_OK;
}

int bnn_survival_instability(const float* d_t, int64_t n_systems, int32_t n_trios, int64_t n_units,
                             const float* h_thresholds, int32_t n_thresholds, float* d_surv, void* stream) {
    using namespace bnn;
    // argument checks first: they need no device
    BNN_REQUIRE(d_t && h_thresholds && d_surv && n_systems > 0 && n_units > 0 && n_trios >= 1, BNN_E_ARG,
                "bnn_survival_instability: null pointer or empty problem");
    SurvivalThresholds th;
    int rc = survival_thresholds("bnn_survival_instability", h_thresholds, n_thresholds, th);
    if (rc != BNN_OK) return rc;
    BNN_REQUIRE(n_systems < (1ll << 31) && n_units < (1ll << 32), BNN_E_ARG,
                "bnn_survival_instability: n_systems must be < 2^31 and n_units < 2^32");
    BNN_REQUIRE(aligned(d_t, 4) && aligned(d_surv, 4), BNN_E_ALIGN, "bnn_survival_instability: pointers must be 4-byte aligned");
    rc = check_device();
    if (rc != BNN_OK) return rc;
    survival_kernel<<<(unsigned)n_systems, SURV_THREADS, 0, (cudaStream_t)stream>>>(d_t, UniformRows{n_trios}, n_units, th,
                                                                                     d_surv);
    BNN_CUDA(cudaGetLastError());
    return BNN_OK;
}

int bnn_survival_instability_ragged(const float* d_t, int64_t n_systems, const int64_t* d_row_offsets, int64_t n_units,
                                    const float* h_thresholds, int32_t n_thresholds, float* d_surv, void* stream) {
    using namespace bnn;
    // argument checks first: they need no device
    BNN_REQUIRE(d_t && h_thresholds && d_surv && d_row_offsets && n_systems > 0 && n_units > 0, BNN_E_ARG,
                "bnn_survival_instability_ragged: null pointer or empty problem");
    SurvivalThresholds th;
    int rc = survival_thresholds("bnn_survival_instability_ragged", h_thresholds, n_thresholds, th);
    if (rc != BNN_OK) return rc;
    BNN_REQUIRE(n_systems < (1ll << 31) && n_units < (1ll << 32), BNN_E_ARG,
                "bnn_survival_instability_ragged: n_systems must be < 2^31 and n_units < 2^32");
    BNN_REQUIRE(aligned(d_t, 4) && aligned(d_surv, 4), BNN_E_ALIGN,
                "bnn_survival_instability_ragged: pointers must be 4-byte aligned");
    BNN_REQUIRE(aligned(d_row_offsets, 8), BNN_E_ALIGN, "bnn_survival_instability_ragged: d_row_offsets must be 8-byte aligned");
    rc = check_device();
    if (rc != BNN_OK) return rc;
    survival_kernel<<<(unsigned)n_systems, SURV_THREADS, 0, (cudaStream_t)stream>>>(d_t, RaggedRows{d_row_offsets}, n_units,
                                                                                     th, d_surv);
    BNN_CUDA(cudaGetLastError());
    return BNN_OK;
}

int bnn_first_trio_instability(const float* d_t, int64_t n_systems, int32_t n_trios, int64_t n_units, float* d_first,
                               void* stream) {
    using namespace bnn;
    // argument checks first: they need no device
    BNN_REQUIRE(d_t && d_first && n_systems > 0 && n_units > 0 && n_trios >= 1, BNN_E_ARG,
                "bnn_first_trio_instability: null pointer or empty problem");
    BNN_REQUIRE(n_trios <= FIRST_MAXR, BNN_E_ARG, "bnn_first_trio_instability: %d trios per system, at most %d supported",
                (int)n_trios, FIRST_MAXR);
    BNN_REQUIRE(n_systems < (1ll << 31) && n_units < (1ll << 32), BNN_E_ARG,
                "bnn_first_trio_instability: n_systems must be < 2^31 and n_units < 2^32");
    BNN_REQUIRE(aligned(d_t, 4) && aligned(d_first, 4), BNN_E_ALIGN,
                "bnn_first_trio_instability: pointers must be 4-byte aligned");
    int rc = check_device();
    if (rc != BNN_OK) return rc;
    first_trio_kernel<<<(unsigned)n_systems, FIRST_THREADS, 0, (cudaStream_t)stream>>>(d_t, UniformRows{n_trios}, n_units,
                                                                                        d_first);
    BNN_CUDA(cudaGetLastError());
    return BNN_OK;
}

int bnn_first_trio_instability_ragged(const float* d_t, int64_t n_systems, const int64_t* d_row_offsets, int64_t n_units,
                                      float* d_first, void* stream) {
    using namespace bnn;
    // argument checks first: they need no device
    BNN_REQUIRE(d_t && d_first && d_row_offsets && n_systems > 0 && n_units > 0, BNN_E_ARG,
                "bnn_first_trio_instability_ragged: null pointer or empty problem");
    BNN_REQUIRE(n_systems < (1ll << 31) && n_units < (1ll << 32), BNN_E_ARG,
                "bnn_first_trio_instability_ragged: n_systems must be < 2^31 and n_units < 2^32");
    BNN_REQUIRE(aligned(d_t, 4) && aligned(d_first, 4), BNN_E_ALIGN,
                "bnn_first_trio_instability_ragged: pointers must be 4-byte aligned");
    BNN_REQUIRE(aligned(d_row_offsets, 8), BNN_E_ALIGN,
                "bnn_first_trio_instability_ragged: d_row_offsets must be 8-byte aligned");
    int rc = check_device();
    if (rc != BNN_OK) return rc;
    first_trio_kernel<<<(unsigned)n_systems, FIRST_THREADS, 0, (cudaStream_t)stream>>>(d_t, RaggedRows{d_row_offsets},
                                                                                        n_units, d_first);
    BNN_CUDA(cudaGetLastError());
    return BNN_OK;
}

int bnn_decompose_uncertainty(const float* d_pred, int64_t n_rows, int64_t n_units, int64_t units_per_model,
                              float* d_out, void* stream) {
    using namespace bnn;
    // argument checks first: they need no device
    BNN_REQUIRE(d_pred && d_out && n_rows > 0 && n_units > 0, BNN_E_ARG,
                "bnn_decompose_uncertainty: null pointer or empty problem");
    BNN_REQUIRE(n_rows < (1ll << 31) && n_units < (1ll << 32), BNN_E_ARG,
                "bnn_decompose_uncertainty: n_rows must be < 2^31 and n_units < 2^32");
    BNN_REQUIRE(units_per_model >= 1 && n_units % units_per_model == 0, BNN_E_ARG,
                "bnn_decompose_uncertainty: n_units (%lld) must be a positive multiple of units_per_model (%lld)",
                (long long)n_units, (long long)units_per_model);
    const int64_t n_models = n_units / units_per_model;
    BNN_REQUIRE(n_models <= UNC_MAXM, BNN_E_ARG, "bnn_decompose_uncertainty: %lld models, at most %d supported",
                (long long)n_models, UNC_MAXM);
    BNN_REQUIRE((reinterpret_cast<uintptr_t>(d_pred) & 7u) == 0 && (reinterpret_cast<uintptr_t>(d_out) & 3u) == 0,
                BNN_E_ALIGN, "bnn_decompose_uncertainty: d_pred must be 8-byte and d_out 4-byte aligned");
    int rc = check_device();
    if (rc != BNN_OK) return rc;
    static PerDeviceOnce attr_done;
    if (attr_done.need()) {
        BNN_CUDA(cudaFuncSetAttribute(uncertainty_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)(UNC_WARPS * UNC_MAXM * sizeof(double))));
    }
    const size_t smem = (size_t)UNC_WARPS * n_models * sizeof(double);
    uncertainty_kernel<<<(unsigned)n_rows, UNC_THREADS, smem, (cudaStream_t)stream>>>(
        (const float2*)d_pred, n_units, (uint32_t)units_per_model, (int)n_models, d_out);
    BNN_CUDA(cudaGetLastError());
    return BNN_OK;
}

}  // extern "C"

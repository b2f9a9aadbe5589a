// K4: fused SWAG training step -- noisy forward + analytic backward + clip + SGD-momentum or Adam for n_seeds
// independent models in one call, and the validation loss (bnn_eval_loss).
//
// Reference: SWAGModel.training_step (/root/reference/spock_reg_model.py:722-732) -> lossfnc (:579-583) ->
// VarModel.forward(noisy_val=True) (:486-528) -> _lossfnc (:547-577); loss.backward(); Lightning's
// gradient_clip_val = clip_grad_norm_ (run_swag.py:61,74-79); torch.optim.SGD(momentum, weight_decay) (:709-711).
//
// total = sum_b nll_b + beta_in * B * 1/2 sum_c (e^{lvin_c} - lvin_c - 1) + beta_out * sum_{b,j} 1/2 (s_bj^2 + e^{lvs_j} - lvs_j - 1)
//
// Backward (per system; T rows, n = T), derived by hand and checked against the reference's autograd gradient
// (tests/golden/train_v50.npz):
//   head:   g_r = (g_mu * (hi-lo)/2 (1 - tanh^2 r0), g_sd * ...);  dV2 += g_r r2^T;  g_a2 = (V2^T g_r) . [r2>0];
//           dV1 += g_a2 r1^T;  g_a1 = (V1^T g_a2) . [r1>0];  dV0 += g_a1 s'^T;  g_s' = V0^T g_a1
//   noise:  s' = s + eps_sum e^{lvs/2}:  g_s = g_s' + beta_out s;  dlvs += g_s' (s'-s)/2  (+ beta_out B (e^{lvs}-1)/2)
//   stats:  s = [mu_s, sqrt(|v_s|+1e-5)], mu_s = eps1 sqrt(v/n) + m, v_s = eps2 sqrt(2 v^2/(n-1)) + v:
//           g_m = g_mus;  g_v = g_mus eps1 / (2 n sqrt(v/n)) + g_vs (1 + eps2 2 v / ((n-1) sqrt(2 v^2/(n-1)))),
//           g_vs = g_sds sign(v_s) / (2 sd_s);   g_f[t] = g_m / n + g_v 2 (f_t - m) / (n-1)      (v = std^2, unbiased)
//   MLP:    dW2 += g_f^T h2; g_a2 = (g_f W2) . [h2>0]; dW1 += g_a2^T h1; g_a1 = (g_a2 W1) . [h1>0]; dW0 += g_a1^T x';
//           g_x = g_a1 W0;  x' = mask(x) + eps_in e^{lvin/2}:  dlvin += g_x . (x' - mask(x)) / 2  (+ beta_in B (e^{lvin}-1)/2)
//
// Decomposition: one CTA owns a seed and walks that seed's systems (grid = n_cta x n_seeds); a system's T x 41
// input, both hidden activations and the latent rows stay in shared memory (feature-major [feature][row]) for the
// whole forward + backward; every thread accumulates its own block of every weight gradient in registers over all
// systems of the CTA, writes one partial gradient vector per CTA, and a second kernel adds the partials in a fixed
// order (bit-reproducible SWAG moments), a third computes the global norm, clips and applies SGD (bnn_train_step) or
// Adam (bnn_train_step_adam).
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "loss_device.cuh"
#include "predict_device.cuh"

namespace bnn {
namespace train {

constexpr int DPAD = 8;            // metric slots appended to each gradient partial
constexpr int SLOT_NLL = 0, SLOT_SKL = 1;

struct Params {
    const float* theta;        // [n_seeds, d]
    const float* X;            // [n_data, T, F]
    const float* Y;            // [n_data, 2]
    const int32_t* batch_index;  // [n_seeds, B] rows of X / Y, or null (row = b)
    const float* eps_in;       // [n_seeds, B, T, F] or null
    const float* eps12;        // [n_seeds, B, 2L] or null
    const float* eps_sum;      // [n_seeds, B, 2L] or null
    float* partial;            // [n_seeds, n_cta, d + DPAD]
    float* head_rec;           // [n_seeds, B, REC] per-system head vectors (v3 only)
    float* xprod;              // [n_seeds, n_cta, 2, 2, F, 2T] input-tile scratch of the producer warps (v3 only)
    int saliency;              // v3 only: d mu / d x instead of the training gradient (bnn_saliency)
    float* gx_out;             // [n_seeds, B, T, F] or null
    float* mu_out;             // [n_seeds, B]
    int B, T, F, FP, n_cta;
    int seed0;                 // first seed of this launch: seed index = seed0 + blockIdx.y (seed groups, see pick_plan)
    uint64_t seed, step;
    uint64_t zero_mask;
    HeadConsts hc;
    float beta_out;
};

// Philox key of one seed-model's noise streams; counters: (block, batch position, step, stream)
__host__ __device__ inline uint64_t seed_key(uint64_t seed, int seed_index) {
    return seed + 0x9E3779B97F4A7C15ull * (uint64_t)(seed_index + 1);
}

}  // namespace train
}  // namespace bnn
#include "train_v3.cuh"
#include "train_tc.cuh"
namespace bnn {
namespace train {

// grad[s][i] = sum_c partial[s][c][i] (fixed order) + analytic KL terms; per-block sum of squares.
__global__ void __launch_bounds__(256) train_reduce_kernel(const float* __restrict__ partial, const float* __restrict__ theta,
                                                           int n_cta, int d, int F, float kl_in_scale, float kl_sum_scale,
                                                           float* __restrict__ grad, float* __restrict__ sq) {
    __shared__ float sh[256];
    const int s = blockIdx.y, i = blockIdx.x * 256 + threadIdx.x;
    const int DP = d + DPAD;
    float g = 0.f;
    if (i < DP) {
        const float* p = partial + (int64_t)s * n_cta * DP + i;
        for (int c = 0; c < n_cta; ++c) g += p[(int64_t)c * DP];
        if (i < F) {  // input_kl * beta_in * B (:585-590, :726): d/dlv = (e^lv - 1)/2
            g += kl_in_scale * 0.5f * (expf(theta[(int64_t)s * d + i]) - 1.0f);
        } else if (i < F + S2) {  // summary_kl * beta_out, summed over the batch (:515-520, :727)
            g += kl_sum_scale * 0.5f * (expf(theta[(int64_t)s * d + i]) - 1.0f);
        }
        grad[(int64_t)s * DP + i] = g;
    }
    sh[threadIdx.x] = (i < d) ? g * g : 0.f;
    __syncthreads();
    for (int st = 128; st > 0; st >>= 1) {
        if ((int)threadIdx.x < st) sh[threadIdx.x] += sh[threadIdx.x + st];
        __syncthreads();
    }
    if (threadIdx.x == 0) sq[s * gridDim.x + blockIdx.x] = sh[0];
}

// Prologue of both update kernels: clip_grad_norm_ over seed s's whole gradient (coef = clip / (norm + 1e-6), applied
// when < 1), grad_out and the metric slots known from the gradient.  Returns the factor the gradient is scaled by
// (min(1, coef)) and this thread's gradient element in gi (0 past d).
__device__ __forceinline__ float clip_prologue(const float* __restrict__ grad, const float* __restrict__ sq, int n_blocks,
                                               int d, int B, const bnn_train_hparams& hp, float* __restrict__ grad_out,
                                               float* __restrict__ metrics, float& gi) {
    const int s = blockIdx.y, i = blockIdx.x * 256 + threadIdx.x;
    float ss = 0.f;
    for (int b = 0; b < n_blocks; ++b) ss += sq[s * n_blocks + b];
    const float norm = sqrtf(ss);
    const float coef = hp.clip_norm / (norm + 1e-6f);
    const float clip = coef < 1.0f ? coef : 1.0f;
    const float* g = grad + (int64_t)s * (d + DPAD);
    gi = i < d ? g[i] : 0.f;
    if (grad_out && i < d) grad_out[(int64_t)s * d + i] = gi;
    if (metrics && blockIdx.x == gridDim.x - 1 && threadIdx.x == 255) {
        float* m = metrics + s * 8;
        const float nll = g[d + SLOT_NLL], skl = g[d + SLOT_SKL] * hp.beta_out;
        m[0] = nll / (float)B;
        m[3] = skl / (float)B;
        m[4] = norm;
        m[5] = clip;
        m[6] = isfinite(nll + skl + norm) ? 0.f : 1.f;
        m[7] = 0.f;
        // m[1] (loss with reg) and m[2] (input_kl) are completed by train_metrics_kernel, which reads lv_in before the update
    }
    return clip;
}

// clip_grad_norm_ + torch.optim.SGD with momentum / weight decay.
__global__ void __launch_bounds__(256) train_update_kernel(const float* __restrict__ grad, const float* __restrict__ sq,
                                                           int n_blocks, int d, int B, bnn_train_hparams hp,
                                                           float* __restrict__ theta, float* __restrict__ mom,
                                                           float* __restrict__ grad_out, float* __restrict__ metrics) {
    const int s = blockIdx.y, i = blockIdx.x * 256 + threadIdx.x;
    float gi;
    const float clip = clip_prologue(grad, sq, n_blocks, d, B, hp, grad_out, metrics, gi);
    if (i < d && hp.apply_update) {
        const int64_t o = (int64_t)s * d + i;
        const float th = theta[o];
        float dp = gi * clip;   // clip == 1 when not clipping: exact
        if (hp.weight_decay != 0.f) dp = fmaf(hp.weight_decay, th, dp);
        const float buf = hp.first_step ? dp : fmaf(hp.momentum, mom[o], dp);
        mom[o] = buf;
        theta[o] = th - hp.lr * buf;
    }
}

// The per-step scalars of torch.optim.Adam, computed on the host in double (torch's Python floats) and cast once.
struct AdamStep {
    float step_size;   // lr / (1 - beta1^t), beta1 of THIS step (the one-cycle schedule cycles it)
    float bc2_sqrt;    // sqrt(1 - beta2^t)
    float w1;          // 1 - beta1: exp_avg.lerp_(g, 1 - beta1)
    float beta2, w2;   // beta2, 1 - beta2: exp_avg_sq.mul_(beta2).addcmul_(g, g, value=1 - beta2)
    float eps;
    int first;         // t == 1: both buffers are zero and are not read (a fresh optimizer; no memset needed)
};

// clip_grad_norm_ + torch.optim.Adam (amsgrad=False, maximize=False; weight decay is L2 added to the gradient, not AdamW):
//   g += wd theta;  m = lerp(m, g, 1 - beta1);  v = beta2 v + (1 - beta2) g^2;  theta -= step_size m / (sqrt(v) / bc2_sqrt + eps)
__global__ void __launch_bounds__(256) train_adam_update_kernel(const float* __restrict__ grad, const float* __restrict__ sq,
                                                                int n_blocks, int d, int B, bnn_train_hparams hp, AdamStep a,
                                                                float* __restrict__ theta, float* __restrict__ exp_avg,
                                                                float* __restrict__ exp_avg_sq, float* __restrict__ grad_out,
                                                                float* __restrict__ metrics) {
    const int s = blockIdx.y, i = blockIdx.x * 256 + threadIdx.x;
    float gi;
    const float clip = clip_prologue(grad, sq, n_blocks, d, B, hp, grad_out, metrics, gi);
    if (i < d && hp.apply_update) {
        const int64_t o = (int64_t)s * d + i;
        const float th = theta[o];
        float g = gi * clip;
        if (hp.weight_decay != 0.f) g = fmaf(hp.weight_decay, th, g);
        const float m0 = a.first ? 0.f : exp_avg[o], v0 = a.first ? 0.f : exp_avg_sq[o];
        const float diff = g - m0;   // torch's lerp: from the nearer end of the weight
        const float m = a.w1 < 0.5f ? fmaf(a.w1, diff, m0) : fmaf(-diff, 1.0f - a.w1, g);
        const float v = fmaf(a.w2 * g, g, v0 * a.beta2);
        exp_avg[o] = m;
        exp_avg_sq[o] = v;
        theta[o] = th - a.step_size * (m / (sqrtf(v) / a.bc2_sqrt + a.eps));
    }
}

// input_kl * beta_in * B / B and the total, from the weights the step was evaluated at (runs BEFORE the update kernel)
__global__ void train_metrics_kernel(const float* __restrict__ theta, const float* __restrict__ grad, int d, int F, int B,
                                     bnn_train_hparams hp, float* __restrict__ metrics) {
    const int s = blockIdx.x;
    if (threadIdx.x != 0) return;
    float kl = 0.f;
    for (int c = 0; c < F; ++c) {
        const float lv = theta[(int64_t)s * d + c];
        kl += expf(lv) - lv - 1.0f;
    }
    const float ikl = 0.5f * kl * hp.beta_in * (float)B;
    const float* g = grad + (int64_t)s * (d + DPAD);
    const float nll = g[d + SLOT_NLL], skl = g[d + SLOT_SKL] * hp.beta_out;
    metrics[s * 8 + 1] = (nll + (ikl + skl)) / (float)B;
    metrics[s * 8 + 2] = ikl / (float)B;
}

// the Philox draws of one training step, written out (parity tests feed them to the oracle)
// tc_map: the tensor-core kernel's producers draw per (row quad q, column c) -- block q * F + c gives rows 4q..4q+3 of
// column c -- where the FFMA kernel draws per (row t, 4-column group); the two kernels see different noise for the
// same (seed, step), each equal to what this kernel writes for its mapping.
__global__ void train_noise_kernel(int B, int T, int F, uint64_t seed, uint64_t step, int tc_map, float* __restrict__ eps_in,
                                   float* __restrict__ eps12, float* __restrict__ eps_sum) {
    const int sidx = blockIdx.y, b = blockIdx.x;
    const uint64_t key = seed_key(seed, sidx);
    const int64_t sb = (int64_t)sidx * B + b;
    const int F4 = (F + 3) >> 2;
    if (tc_map) {
        for (int i = threadIdx.x; i < (T / 4) * F; i += blockDim.x) {
            const int q = i / F, c = i - q * F;
            const float4 n4 = philox_normal4_fast(key, STREAM_EPS_IN, (uint32_t)b, (uint32_t)step, (uint32_t)i);
            const float e[4] = {n4.x, n4.y, n4.z, n4.w};
            for (int u = 0; u < 4; ++u) eps_in[(sb * T + 4 * q + u) * F + c] = e[u];
        }
    } else
    for (int i = threadIdx.x; i < T * F4; i += blockDim.x) {
        const int t = i / F4, c4 = i - t * F4;
        const float4 n4 = philox_normal4_fast(key, STREAM_EPS_IN, (uint32_t)b, (uint32_t)step, (uint32_t)i);
        const float e[4] = {n4.x, n4.y, n4.z, n4.w};
        for (int u = 0; u < 4; ++u)
            if (4 * c4 + u < F) eps_in[(sb * T + t) * F + 4 * c4 + u] = e[u];
    }
    if (threadIdx.x < S2 / 4) {
        reinterpret_cast<float4*>(eps12 + sb * S2)[threadIdx.x] =
            philox_normal4(key, STREAM_EPS, (uint32_t)b, (uint32_t)step, threadIdx.x);
        reinterpret_cast<float4*>(eps_sum + sb * S2)[threadIdx.x] =
            philox_normal4(key, STREAM_EPS_SUM, (uint32_t)b, (uint32_t)step, threadIdx.x);
    }
}

// loss_sum[u] = sum_b _lossfnc(out[u][b], y[b]) -- one block per unit, fixed order
__global__ void __launch_bounds__(256) nll_sum_kernel(const float2* __restrict__ out, const float2* __restrict__ y, int64_t B,
                                                      float* __restrict__ loss_sum) {
    __shared__ float sh[256];
    const float2* o = out + (int64_t)blockIdx.x * B;
    float acc = 0.f;
    for (int64_t b = threadIdx.x; b < B; b += 256) {
        float l0, l1, a, c;
        const float2 p = o[b], yy = y[b];
        nll_terms(p.x, p.y, yy.x, l0, a, c);
        nll_terms(p.x, p.y, yy.y, l1, a, c);
        acc += -(l0 + l1);
    }
    sh[threadIdx.x] = acc;
    __syncthreads();
    for (int st = 128; st > 0; st >>= 1) {
        if ((int)threadIdx.x < st) sh[threadIdx.x] += sh[threadIdx.x + st];
        __syncthreads();
    }
    if (threadIdx.x == 0) loss_sum[blockIdx.x] = sh[0];
}

// sumsq[s][c] = sum over the CTAs' partial sums of (d mu / d x)^2 in column c (the v3 kernel parks them, halved, in the
// dlv_in slot of its partial), fixed order
__global__ void saliency_finish_kernel(const float* __restrict__ partial, int n_cta, int d, int F, float* __restrict__ sumsq) {
    const int s = blockIdx.x, c = threadIdx.x;
    if (c >= F) return;
    const float* p = partial + (int64_t)s * n_cta * (d + DPAD) + c;
    float a = 0.f;
    for (int i = 0; i < n_cta; ++i) a += p[(int64_t)i * (d + DPAD)];
    sumsq[s * F + c] = 2.0f * a;
}

// Kernel selection.  Default: the tensor-core kernel (train_tc.cuh) when the shape is the reference's (T = 100, F = 41)
// and the input image of the flag set fits its shared-memory plan (every shipped checkpoint: 31 live columns); else the
// FP32 FFMA kernel (train_v3.cuh).  A process-wide override for tests / tools: bnn_set_train_variant() (diagnostic
// header), initialised ONCE from the environment variable BNN_TRAIN_VARIANT = tc | v3.
enum { VARIANT_AUTO = 0, VARIANT_TC = 1, VARIANT_V3 = 2 };
static int g_train_variant = -1;
static int train_variant() {
    if (g_train_variant < 0) {
        const char* force = getenv("BNN_TRAIN_VARIANT");
        g_train_variant = !force ? VARIANT_AUTO : (!strcmp(force, "tc") ? VARIANT_TC : (!strcmp(force, "v3") ? VARIANT_V3 : VARIANT_AUTO));
    }
    return g_train_variant;
}
static bool shape_ok(const bnn_model_config* cfg) { return cfg->n_times == 100 && cfg->n_features == 41; }
// Automatic selection also asks for B >= TC_MIN_BATCH: the weight-gradient GEMMs of the tensor-core kernel are single-pass
// TF32 on round-to-nearest operands, whose unbiased rounding noise falls as 1 / sqrt(B T); at B = 2000 the gradient matches
// the fp32 reference to 3e-6 of its max-norm (theta after a step to 1e-7), at B = 32..64 to 2e-5 (theta 1e-6), where
// the FP32 kernel keeps the 1e-6 / 1e-7 parity -- and such batches cannot fill the GPU anyway.
constexpr int64_t TC_MIN_BATCH = 256;
static bool use_tc(const bnn_model_config* cfg, int64_t B) {
    if (!shape_ok(cfg) || train_variant() == VARIANT_V3) return false;
    if (train_variant() == VARIANT_AUTO && B < TC_MIN_BATCH) return false;
    return tcx::SmemTC(cfg->zero_mask).fits();
}

// per-CTA input-tile scratch in the workspace: v3's two parities of (x' | n | small inputs), or the tensor-core kernel's
// ring of NST images
static size_t scratch_floats_per_cta(const bnn_model_config* cfg) {
    const size_t v3 = (size_t)8 * cfg->n_features * cfg->n_times + 2 * XSM;
    const size_t tc = (size_t)tcx::NST * (tcx::NQ * 97 * 4 + tcx::SMALLF + tcx::XG * 4 * tcx::NQ * 4);
    return v3 > tc ? v3 : tc;
}

static int sm_count() {
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess ||
        sms < 1) {
        cudaGetLastError();   // no device (host-only plan queries): a B200's SM count
        sms = 148;
    }
    return sms;
}

// One CTA per SM, never more CTAs than SMs (a 149th CTA would run alone in a second wave); a seed's CTAs walk its
// systems (tc: one per tile, v3: two per iteration).  A CTA belongs to ONE seed (its weights live in shared memory, its
// weight-gradient accumulators in tensor memory), so with n_seeds CTAs-per-seed = floor(SMs / n_seeds) can leave many SMs
// idle: 30 seeds -> 4 CTAs each = 120 of 148 SMs, 500 systems per CTA.  The seeds are therefore run in `groups` launches of
// `per` seeds each when that shortens the step: 3 launches of 10 seeds x 14 CTAs walk 143 systems per CTA each (429 in all).
// Cost model: systems per CTA + ~4 systems' worth of fixed cost per launch (prologue, pipeline fill, partial write-out).
struct SeedPlan { int n_cta, groups, per; };
static int g_seed_groups = 0;   // bnn_set_train_seed_groups (diagnostic header): 0 = cost model, g = that many groups
static SeedPlan pick_plan(const bnn_model_config* cfg, int64_t B, int n_seeds) {
    const int64_t sms = sm_count();
    const int64_t cap = use_tc(cfg, B) ? B : (B + 1) / 2;
    SeedPlan best{1, 1, n_seeds};
    double best_cost = 0.0;
    const int g_lo = g_seed_groups > 0 ? (g_seed_groups < n_seeds ? g_seed_groups : n_seeds) : 1;
    const int g_hi = g_seed_groups > 0 ? g_lo : 8;
    for (int g = g_lo; g <= g_hi && g <= n_seeds; ++g) {
        const int per = (n_seeds + g - 1) / g;
        const int groups = (n_seeds + per - 1) / per;
        int64_t n = sms / per;
        if (n > cap) n = cap;
        if (n < 1) n = 1;
        const double cost = groups * ((double)((B + n - 1) / n) + 4.0);
        if (g == g_lo || cost < 0.95 * best_cost) { best = SeedPlan{(int)n, groups, per}; best_cost = cost; }
    }
    return best;
}
static int pick_n_cta(const bnn_model_config* cfg, int64_t B, int n_seeds) { return pick_plan(cfg, B, n_seeds).n_cta; }

// Everything of a training step before the optimizer's update, shared by bnn_train_step (SGD) and bnn_train_step_adam:
// the argument checks (`who` names the entry in messages; `state_ok`: the optimizer's state buffers are given, required
// when hp->apply_update), the seed-group launches of the training kernel, the fixed-order reduce and the logged metrics.
// On BNN_OK the reduced gradient and its per-block sums of squares are enqueued on st for the update kernel.
struct Gradient { const float* grad; const float* sq; int nb, d; };
static int train_gradient(const char* who, bool state_ok, const char* state_name, const bnn_model_config* cfg,
                          const bnn_train_hparams* hp, int32_t n_seeds, const float* d_theta, const float* d_x,
                          const float* d_y, const int32_t* d_batch_index, int64_t B, const float* d_eps_in,
                          const float* d_eps12, const float* d_eps_sum, uint64_t seed, uint64_t step, float* d_metrics,
                          void* d_workspace, cudaStream_t st, Gradient* out) {
    int rc = validate_config(cfg);
    if (rc != BNN_OK) return rc;
    if ((rc = check_device()) != BNN_OK) return rc;
    BNN_REQUIRE(hp && d_theta && d_x && d_y && d_workspace, BNN_E_ARG, "%s: null pointer", who);
    BNN_REQUIRE(n_seeds >= 1 && n_seeds <= 65535 && B >= 1 && B < (1ll << 30), BNN_E_ARG,
                "%s: n_seeds=%d B=%lld out of range", who, n_seeds, (long long)B);
    BNN_REQUIRE(!hp->apply_update || state_ok, BNN_E_ARG, "%s: %s required to update", who, state_name);
    const bool any = d_eps_in || d_eps12 || d_eps_sum, all = d_eps_in && d_eps12 && d_eps_sum;
    BNN_REQUIRE(!any || all, BNN_E_ARG, "%s: give all of eps_in, eps12, eps_sum or none", who);
    BNN_REQUIRE(aligned16(d_workspace) && (!d_eps12 || (aligned16(d_eps12) && aligned16(d_eps_sum))), BNN_E_ALIGN,
                "%s: workspace / eps12 / eps_sum must be 16-byte aligned", who);
    const int F = cfg->n_features, T = cfg->n_times, FP = (F + 3) & ~3;
    BNN_REQUIRE(shape_ok(cfg), BNN_E_CONFIG, "%s: compiled for the reference's shape T=100, F=41 (got T=%d, F=%d)", who, T, F);
    const FlatLayout fl(F);
    const SeedPlan plan = pick_plan(cfg, B, n_seeds);
    const int n_cta = plan.n_cta;
    const int DP = fl.d + DPAD, nb = (DP + 255) / 256;
    float* partial = (float*)d_workspace;
    float* grad = partial + (size_t)n_seeds * n_cta * DP;
    float* sq = grad + (size_t)n_seeds * DP;
    float* head_rec = sq + (size_t)n_seeds * nb;
    head_rec += (4 - ((uintptr_t)head_rec / sizeof(float)) % 4) % 4;  // 16-byte aligned records

    Params prm;
    prm.theta = d_theta; prm.X = d_x; prm.Y = d_y; prm.batch_index = d_batch_index;
    prm.eps_in = d_eps_in; prm.eps12 = d_eps12; prm.eps_sum = d_eps_sum;
    prm.partial = partial;
    prm.head_rec = head_rec;
    prm.xprod = head_rec + (size_t)n_seeds * B * REC;   // REC is a multiple of 4: stays 16-byte aligned
    prm.B = (int)B; prm.T = T; prm.F = F; prm.FP = FP; prm.n_cta = n_cta; prm.seed0 = 0;
    prm.seed = seed; prm.step = step; prm.zero_mask = cfg->zero_mask;
    prm.hc = HeadConsts{cfg->lo_mu, cfg->hi_mu, cfg->lo_sd, cfg->hi_sd};
    prm.beta_out = hp->beta_out;
    prm.saliency = 0; prm.gx_out = nullptr; prm.mu_out = nullptr;
    if (use_tc(cfg, B)) {
        const size_t smem_tc = (size_t)tcx::SmemTC(cfg->zero_mask).total * sizeof(float);
        static PerDeviceOnce attr_tc_done;
        if (attr_tc_done.need()) {
            BNN_CUDA(cudaFuncSetAttribute(train_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        }
        for (int s0 = 0; s0 < n_seeds; s0 += plan.per) {   // seed groups (pick_plan); every buffer is indexed by the global seed
            prm.seed0 = s0;
            train_tc_kernel<<<dim3(n_cta, n_seeds - s0 < plan.per ? n_seeds - s0 : plan.per), tcx::NTHR_TC, smem_tc, st>>>(prm);
        }
    } else {
        const size_t smem3 = (size_t)Smem3(T, F).total * sizeof(float);
        static PerDeviceOnce attr3_done;
        if (attr3_done.need()) {
            BNN_CUDA(cudaFuncSetAttribute(train_fwd_bwd3_kernel<100, 41>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          227 * 1024));
        }
        for (int s0 = 0; s0 < n_seeds; s0 += plan.per) {
            prm.seed0 = s0;
            train_fwd_bwd3_kernel<100, 41><<<dim3(n_cta, n_seeds - s0 < plan.per ? n_seeds - s0 : plan.per), NTHR3, smem3, st>>>(
                prm);
        }
    }
    BNN_CUDA(cudaGetLastError());
    train_reduce_kernel<<<dim3(nb, n_seeds), 256, 0, st>>>(partial, d_theta, n_cta, fl.d, F, hp->beta_in * (float)B,
                                                          hp->beta_out * (float)B, grad, sq);
    BNN_CUDA(cudaGetLastError());
    if (d_metrics) {
        train_metrics_kernel<<<n_seeds, 32, 0, st>>>(d_theta, grad, fl.d, F, (int)B, *hp, d_metrics);
        BNN_CUDA(cudaGetLastError());
    }
    *out = Gradient{grad, sq, nb, fl.d};
    return BNN_OK;
}

}  // namespace train
}  // namespace bnn

extern "C" {

size_t bnn_train_workspace_bytes(const bnn_model_config* cfg, int64_t B, int32_t n_seeds) {
    using namespace bnn;
    if (validate_config(cfg) != BNN_OK || B <= 0 || n_seeds <= 0) return 0;
    const int d = FlatLayout(cfg->n_features).d;
    const int n_cta = train::pick_n_cta(cfg, B, n_seeds);
    const size_t DP = d + train::DPAD;
    const size_t nb = (DP + 255) / 256;
    // partial | grad | sq | pad | head records (v3)
    return ((size_t)n_seeds * n_cta * DP + (size_t)n_seeds * DP + (size_t)n_seeds * nb + 64 +
            (size_t)n_seeds * B * train::REC + 4 +
            (size_t)n_seeds * n_cta * train::scratch_floats_per_cta(cfg)) * sizeof(float);
}

int bnn_train_step(const bnn_model_config* cfg, const bnn_train_hparams* hp, int32_t n_seeds, float* d_theta,
                   float* d_momentum, const float* d_x, const float* d_y, const int32_t* d_batch_index, int64_t B,
                   const float* d_eps_in, const float* d_eps12, const float* d_eps_sum, uint64_t seed, uint64_t step,
                   float* d_grad_out, float* d_metrics, void* d_workspace, void* stream) {
    using namespace bnn;
    cudaStream_t st = (cudaStream_t)stream;
    train::Gradient gr;
    const int rc = train::train_gradient("bnn_train_step", d_momentum, "momentum buffer", cfg, hp, n_seeds, d_theta, d_x, d_y,
                                        d_batch_index, B, d_eps_in, d_eps12, d_eps_sum, seed, step, d_metrics, d_workspace,
                                        st, &gr);
    if (rc != BNN_OK) return rc;
    train::train_update_kernel<<<dim3(gr.nb, n_seeds), 256, 0, st>>>(gr.grad, gr.sq, gr.nb, gr.d, (int)B, *hp, d_theta,
                                                                    d_momentum, d_grad_out, d_metrics);
    BNN_CUDA(cudaGetLastError());
    return BNN_OK;
}

int bnn_train_step_adam(const bnn_model_config* cfg, const bnn_train_hparams* hp, const bnn_adam_hparams* adam,
                        int32_t n_seeds, float* d_theta, float* d_exp_avg, float* d_exp_avg_sq, const float* d_x,
                        const float* d_y, const int32_t* d_batch_index, int64_t B, const float* d_eps_in,
                        const float* d_eps12, const float* d_eps_sum, uint64_t seed, uint64_t step, float* d_grad_out,
                        float* d_metrics, void* d_workspace, void* stream) {
    using namespace bnn;
    // torch.optim.Adam's constructor checks, written so that NaN fails them too
    BNN_REQUIRE(hp && adam, BNN_E_ARG, "bnn_train_step_adam: null pointer");
    BNN_REQUIRE(hp->lr >= 0.f, BNN_E_ARG, "bnn_train_step_adam: invalid learning rate %g", (double)hp->lr);
    BNN_REQUIRE(hp->weight_decay >= 0.f, BNN_E_ARG, "bnn_train_step_adam: invalid weight_decay %g", (double)hp->weight_decay);
    BNN_REQUIRE(adam->beta1 >= 0.0 && adam->beta1 < 1.0, BNN_E_ARG, "bnn_train_step_adam: invalid beta1 %g (need [0, 1))",
                adam->beta1);
    BNN_REQUIRE(adam->beta2 >= 0.0 && adam->beta2 < 1.0, BNN_E_ARG, "bnn_train_step_adam: invalid beta2 %g (need [0, 1))",
                adam->beta2);
    BNN_REQUIRE(adam->eps >= 0.0, BNN_E_ARG, "bnn_train_step_adam: invalid eps %g", adam->eps);
    BNN_REQUIRE(adam->step >= 1, BNN_E_ARG, "bnn_train_step_adam: step %lld (t is 1-based)", (long long)adam->step);
    cudaStream_t st = (cudaStream_t)stream;
    train::Gradient gr;
    const int rc = train::train_gradient("bnn_train_step_adam", d_exp_avg && d_exp_avg_sq, "exp_avg and exp_avg_sq", cfg, hp,
                                        n_seeds, d_theta, d_x, d_y, d_batch_index, B, d_eps_in, d_eps12, d_eps_sum, seed, step,
                                        d_metrics, d_workspace, st, &gr);
    if (rc != BNN_OK) return rc;
    // bias corrections as torch computes them from Python floats, with this step's beta1
    const double t = (double)adam->step;
    train::AdamStep a;
    a.step_size = (float)((double)hp->lr / (1.0 - pow(adam->beta1, t)));
    a.bc2_sqrt = (float)sqrt(1.0 - pow(adam->beta2, t));
    a.w1 = (float)(1.0 - adam->beta1);
    a.beta2 = (float)adam->beta2;
    a.w2 = (float)(1.0 - adam->beta2);
    a.eps = (float)adam->eps;
    a.first = adam->step == 1;
    train::train_adam_update_kernel<<<dim3(gr.nb, n_seeds), 256, 0, st>>>(gr.grad, gr.sq, gr.nb, gr.d, (int)B, *hp, a,
                                                                         d_theta, d_exp_avg, d_exp_avg_sq, d_grad_out,
                                                                         d_metrics);
    BNN_CUDA(cudaGetLastError());
    return BNN_OK;
}

int bnn_saliency(const bnn_model_config* cfg, int32_t n_models, const float* d_theta, const float* d_x, int64_t B,
                 const float* d_eps12, uint64_t seed, float* d_grad_x, float* d_sumsq, float* d_mu, void* d_workspace,
                 void* stream) {
    using namespace bnn;
    int rc = validate_config(cfg);
    if (rc != BNN_OK) return rc;
    if ((rc = check_device()) != BNN_OK) return rc;
    BNN_REQUIRE(d_theta && d_x && d_sumsq && d_mu && d_workspace, BNN_E_ARG, "bnn_saliency: null pointer");
    BNN_REQUIRE(n_models >= 1 && n_models <= 65535 && B >= 1 && B < (1ll << 30), BNN_E_ARG,
                "bnn_saliency: n_models=%d B=%lld out of range", n_models, (long long)B);
    BNN_REQUIRE(cfg->n_times == 100 && cfg->n_features == 41, BNN_E_CONFIG,
                "bnn_saliency: compiled for T=100, F=41 (got T=%d, F=%d)", cfg->n_times, cfg->n_features);
    BNN_REQUIRE(aligned16(d_workspace) && (!d_eps12 || aligned16(d_eps12)), BNN_E_ALIGN, "bnn_saliency: alignment");
    const int F = cfg->n_features, T = cfg->n_times;
    const FlatLayout fl(F);
    int64_t n_cta = train::sm_count() / n_models;
    if (n_cta > (B + 1) / 2) n_cta = (B + 1) / 2;
    if (n_cta < 1) n_cta = 1;
    const int DP = fl.d + train::DPAD;
    float* partial = (float*)d_workspace;
    float* xprod = partial + (size_t)n_models * n_cta * DP;
    xprod += (4 - ((uintptr_t)xprod / sizeof(float)) % 4) % 4;
    train::Params prm;
    prm.theta = d_theta; prm.X = d_x; prm.Y = nullptr; prm.batch_index = nullptr;
    prm.eps_in = nullptr; prm.eps12 = d_eps12; prm.eps_sum = nullptr;
    prm.partial = partial; prm.head_rec = nullptr; prm.xprod = xprod;
    prm.B = (int)B; prm.T = T; prm.F = F; prm.FP = (F + 3) & ~3; prm.n_cta = (int)n_cta; prm.seed0 = 0;
    prm.seed = seed; prm.step = 0; prm.zero_mask = cfg->zero_mask;
    prm.hc = HeadConsts{cfg->lo_mu, cfg->hi_mu, cfg->lo_sd, cfg->hi_sd};
    prm.beta_out = 0.f;
    prm.saliency = 1; prm.gx_out = d_grad_x; prm.mu_out = d_mu;
    static PerDeviceOnce attr_done;
    if (attr_done.need()) {
        BNN_CUDA(cudaFuncSetAttribute(train::train_fwd_bwd3_kernel<100, 41>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      227 * 1024));
    }
    cudaStream_t st = (cudaStream_t)stream;
    const size_t smem3 = (size_t)train::Smem3(T, F).total * sizeof(float);
    train::train_fwd_bwd3_kernel<100, 41><<<dim3((unsigned)n_cta, n_models), train::NTHR3, smem3, st>>>(prm);
    BNN_CUDA(cudaGetLastError());
    train::saliency_finish_kernel<<<n_models, 64, 0, st>>>(partial, (int)n_cta, fl.d, F, d_sumsq);
    BNN_CUDA(cudaGetLastError());
    return BNN_OK;
}

int bnn_set_train_variant(int32_t variant) {
    using namespace bnn;
    BNN_REQUIRE(variant >= 0 && variant <= 2, BNN_E_ARG, "bnn_set_train_variant: 0 = auto, 1 = tensor-core, 2 = FP32 FFMA (v3)");
    train::g_train_variant = variant;
    return BNN_OK;
}

int bnn_train_seed_plan(const bnn_model_config* cfg, int64_t B, int32_t n_seeds, int32_t* n_cta, int32_t* groups,
                        int32_t* seeds_per_group) {
    using namespace bnn;
    int rc = validate_config(cfg);
    if (rc != BNN_OK) return rc;
    BNN_REQUIRE(B >= 1 && n_seeds >= 1 && n_cta && groups && seeds_per_group, BNN_E_ARG, "bnn_train_seed_plan: bad arguments");
    const train::SeedPlan p = train::pick_plan(cfg, B, n_seeds);
    *n_cta = p.n_cta; *groups = p.groups; *seeds_per_group = p.per;
    return BNN_OK;
}

int bnn_set_train_seed_groups(int32_t groups) {
    using namespace bnn;
    BNN_REQUIRE(groups >= 0 && groups <= 64, BNN_E_ARG, "bnn_set_train_seed_groups: 0 = cost model, 1..64 = launches per step");
    train::g_seed_groups = groups;
    return BNN_OK;
}

int bnn_train_timeline(unsigned long long* host_out, int32_t n) {
    using namespace bnn;
    BNN_REQUIRE(host_out && n >= 0, BNN_E_ARG, "bnn_train_timeline: null pointer");
    for (int i = 0; i < n; ++i) host_out[i] = 0;
#ifdef BNN_TRAIN_TIMELINE
    BNN_CUDA(cudaDeviceSynchronize());
    unsigned long long tmp[train::TL_N];
    BNN_CUDA(cudaMemcpyFromSymbol(tmp, train::g_train_tl, sizeof(tmp)));
    for (int i = 0; i < n && i < train::TL_N; ++i) host_out[i] = tmp[i];
#endif
    return BNN_OK;
}

int bnn_train_noise(const bnn_model_config* cfg, int32_t n_seeds, int64_t B, uint64_t seed, uint64_t step,
                    float* d_eps_in, float* d_eps12, float* d_eps_sum, void* stream) {
    using namespace bnn;
    int rc = validate_config(cfg);
    if (rc != BNN_OK) return rc;
    if ((rc = check_device()) != BNN_OK) return rc;
    BNN_REQUIRE(d_eps_in && d_eps12 && d_eps_sum && n_seeds >= 1 && n_seeds <= 65535 && B >= 1, BNN_E_ARG,
                "bnn_train_noise: null pointer or empty problem");
    BNN_REQUIRE(aligned16(d_eps12) && aligned16(d_eps_sum), BNN_E_ALIGN, "bnn_train_noise: eps12 / eps_sum alignment");
    train::train_noise_kernel<<<dim3((unsigned)B, n_seeds), 128, 0, (cudaStream_t)stream>>>(
        (int)B, cfg->n_times, cfg->n_features, seed, step, train::use_tc(cfg, B) ? 1 : 0, d_eps_in, d_eps12, d_eps_sum);
    BNN_CUDA(cudaGetLastError());
    return BNN_OK;
}

int bnn_eval_loss(const bnn_model_config* cfg, const float* d_x, const float* d_y, int64_t B,
                  const float* d_theta_packed, int64_t n_units, const float* d_eps, uint64_t seed,
                  float* d_out_mu_sd, float* d_loss_sum, void* d_workspace, void* stream) {
    using namespace bnn;
    BNN_REQUIRE(d_y && d_loss_sum, BNN_E_ARG, "bnn_eval_loss: null pointer");
    BNN_REQUIRE(d_out_mu_sd || d_workspace, BNN_E_ARG,
                "bnn_eval_loss: give d_out_mu_sd or a workspace of n_units*B*2 floats");
    BNN_REQUIRE(n_units >= 1 && n_units < (1ll << 31), BNN_E_ARG, "bnn_eval_loss: n_units out of range");
    float* out = d_out_mu_sd ? d_out_mu_sd : (float*)d_workspace;
    int rc = bnn_predict(cfg, d_x, B, d_theta_packed, n_units, d_eps, nullptr, seed, 0, 0, 0, out, nullptr, nullptr, stream);
    if (rc != BNN_OK) return rc;
    train::nll_sum_kernel<<<(unsigned)n_units, 256, 0, (cudaStream_t)stream>>>((const float2*)out, (const float2*)d_y, B,
                                                                              d_loss_sum);
    BNN_CUDA(cudaGetLastError());
    return BNN_OK;
}

}  // extern "C"

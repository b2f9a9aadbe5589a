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
// Per-seed hyperparameters travel in the kernels' parameters (no device copy, no allocation): a launch of the training
// kernel carries the beta_out of at most TRAIN_SEED_CHUNK seeds, a launch of the reduce / update / metrics kernels the
// scalars of at most SEED_CHUNK seeds; larger seed counts are split into launches of that many seeds.
constexpr int TRAIN_SEED_CHUNK = 512;
constexpr int SEED_CHUNK = 64;

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
    float beta_out[TRAIN_SEED_CHUNK];   // of seed seed0 + blockIdx.y (saliency: [0] = 0 for every model)
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

// The scalars of seed s0 + j, in entry j of a launch's SeedChunk (kernel parameters of the reduce / update / metrics
// kernels).  kl_in_scale = beta_in * B and kl_sum_scale = beta_out * B are rounded on the host.
struct SeedHp {
    float lr, momentum, weight_decay, clip_norm, beta_in, beta_out;
    float kl_in_scale, kl_sum_scale;
};
struct SeedChunk { SeedHp s[SEED_CHUNK]; };

// grad[s][i] = sum_c partial[s][c][i] (fixed order) + analytic KL terms; per-block sum of squares.  s = s0 + blockIdx.y.
__global__ void __launch_bounds__(256) train_reduce_kernel(const float* __restrict__ partial, const float* __restrict__ theta,
                                                           int n_cta, int d, int F, int s0, const SeedChunk hp,
                                                           float* __restrict__ grad, float* __restrict__ sq) {
    __shared__ float sh[256];
    const int s = s0 + (int)blockIdx.y, i = blockIdx.x * 256 + threadIdx.x;
    const int DP = d + DPAD;
    float g = 0.f;
    if (i < DP) {
        const float* p = partial + (int64_t)s * n_cta * DP + i;
        for (int c = 0; c < n_cta; ++c) g += p[(int64_t)c * DP];
        if (i < F) {  // input_kl * beta_in * B (:585-590, :726): d/dlv = (e^lv - 1)/2
            g += hp.s[blockIdx.y].kl_in_scale * 0.5f * (expf(theta[(int64_t)s * d + i]) - 1.0f);
        } else if (i < F + S2) {  // summary_kl * beta_out, summed over the batch (:515-520, :727)
            g += hp.s[blockIdx.y].kl_sum_scale * 0.5f * (expf(theta[(int64_t)s * d + i]) - 1.0f);
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
// Per-seed halt (halted_at non-null, the _halt entries): skip is set when seed s is already halted (halted_at[s] >= 0)
// or this step is bad -- nll + skl + norm not finite, the condition of metrics column 6 -- and the thread that writes the
// metrics (the last block's last thread, also when metrics is null) latches halted_at[s] = step when the seed was live.  Every thread of the seed computes the same norm and reads
// the same two metric slots, so it reaches the same decision whichever block runs first: a block that still reads -1
// sees the bad step itself, one that reads the latched word sees a halted seed, and both mean skip.  So the latch needs
// no second kernel and no ordering between blocks.  With halted_at null, skip is false and nothing else changes.
__device__ __forceinline__ float clip_prologue(const float* __restrict__ grad, const float* __restrict__ sq, int n_blocks,
                                               int d, int B, int s, const SeedHp& hp, float* __restrict__ grad_out,
                                               float* __restrict__ metrics, int64_t* halted_at, int64_t step,
                                               float& gi, bool& skip) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    float ss = 0.f;
    for (int b = 0; b < n_blocks; ++b) ss += sq[s * n_blocks + b];
    const float norm = sqrtf(ss);
    const float coef = hp.clip_norm / (norm + 1e-6f);
    const float clip = coef < 1.0f ? coef : 1.0f;
    const float* g = grad + (int64_t)s * (d + DPAD);
    gi = i < d ? g[i] : 0.f;
    if (grad_out && i < d) grad_out[(int64_t)s * d + i] = gi;
    const bool last = blockIdx.x == gridDim.x - 1 && threadIdx.x == 255;
    skip = false;
    if ((metrics && last) || halted_at) {
        const float nll = g[d + SLOT_NLL], skl = g[d + SLOT_SKL] * hp.beta_out;
        const bool bad = !isfinite(nll + skl + norm);
        if (metrics && last) {
            float* m = metrics + s * 8;
            m[0] = nll / (float)B;
            m[3] = skl / (float)B;
            m[4] = norm;
            m[5] = clip;
            m[6] = bad ? 1.f : 0.f;
            m[7] = 0.f;
            // m[1] (loss with reg) and m[2] (input_kl) are completed by train_metrics_kernel, which reads lv_in before the
            // update
        }
        if (halted_at) {
            const bool was = halted_at[s] >= 0;
            skip = was || bad;
            if (last && bad && !was) halted_at[s] = step;
        }
    }
    return clip;
}

// clip_grad_norm_ + torch.optim.SGD with momentum / weight decay.  s = s0 + blockIdx.y.
__global__ void __launch_bounds__(256) train_update_kernel(const float* __restrict__ grad, const float* __restrict__ sq,
                                                           int n_blocks, int d, int B, int s0, const SeedChunk hps,
                                                           int first_step, int apply_update, float* __restrict__ theta,
                                                           float* __restrict__ mom, float* __restrict__ grad_out,
                                                           float* __restrict__ metrics, int64_t* halted_at, int64_t step) {
    const int s = s0 + (int)blockIdx.y, i = blockIdx.x * 256 + threadIdx.x;
    const SeedHp& hp = hps.s[blockIdx.y];
    float gi;
    bool skip;
    const float clip = clip_prologue(grad, sq, n_blocks, d, B, s, hp, grad_out, metrics, halted_at, step, gi, skip);
    if (i < d && apply_update && !skip) {
        const int64_t o = (int64_t)s * d + i;
        const float th = theta[o];
        float dp = gi * clip;   // clip == 1 when not clipping: exact
        if (hp.weight_decay != 0.f) dp = fmaf(hp.weight_decay, th, dp);
        const float buf = first_step ? dp : fmaf(hp.momentum, mom[o], dp);
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
struct AdamChunk { AdamStep a[SEED_CHUNK]; };
// the Adam update kernel's parameters: both chunks, 8 pointers, 5 ints and the step, within the 4 KB every launch may carry
static_assert(sizeof(SeedChunk) + sizeof(AdamChunk) + 8 * 8 + 5 * 4 + 8 <= 4096, "SEED_CHUNK too large for the kernel parameters");

// clip_grad_norm_ + torch.optim.Adam (amsgrad=False, maximize=False; weight decay is L2 added to the gradient, not AdamW):
//   g += wd theta;  m = lerp(m, g, 1 - beta1);  v = beta2 v + (1 - beta2) g^2;  theta -= step_size m / (sqrt(v) / bc2_sqrt + eps)
__global__ void __launch_bounds__(256) train_adam_update_kernel(const float* __restrict__ grad, const float* __restrict__ sq,
                                                                int n_blocks, int d, int B, int s0, const SeedChunk hps,
                                                                const AdamChunk as, int apply_update,
                                                                float* __restrict__ theta, float* __restrict__ exp_avg,
                                                                float* __restrict__ exp_avg_sq, float* __restrict__ grad_out,
                                                                float* __restrict__ metrics, int64_t* halted_at, int64_t step) {
    const int s = s0 + (int)blockIdx.y, i = blockIdx.x * 256 + threadIdx.x;
    const SeedHp& hp = hps.s[blockIdx.y];
    const AdamStep& a = as.a[blockIdx.y];
    float gi;
    bool skip;
    const float clip = clip_prologue(grad, sq, n_blocks, d, B, s, hp, grad_out, metrics, halted_at, step, gi, skip);
    if (i < d && apply_update && !skip) {
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

// input_kl * beta_in * B / B and the total, from the weights the step was evaluated at (runs BEFORE the update kernel).
// s = s0 + blockIdx.x.
__global__ void train_metrics_kernel(const float* __restrict__ theta, const float* __restrict__ grad, int d, int F, int B,
                                     int s0, const SeedChunk hps, float* __restrict__ metrics) {
    const int s = s0 + (int)blockIdx.x;
    if (threadIdx.x != 0) return;
    const SeedHp& hp = hps.s[blockIdx.x];
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

// bytes of the workspace of a step of n_seeds seeds at n_cta CTAs per seed: partial | grad | sq | pad | head records (v3)
// | input-tile scratch
static size_t workspace_bytes(const bnn_model_config* cfg, int64_t B, int32_t n_seeds, int n_cta) {
    const size_t DP = FlatLayout(cfg->n_features).d + DPAD;
    const size_t nb = (DP + 255) / 256;
    return ((size_t)n_seeds * n_cta * DP + (size_t)n_seeds * DP + (size_t)n_seeds * nb + 64 + (size_t)n_seeds * B * REC + 4 +
            (size_t)n_seeds * n_cta * scratch_floats_per_cta(cfg)) * sizeof(float);
}

static SeedChunk seed_chunk(const bnn_train_hparams* hp, int hp_stride, int s0, int n, int64_t B) {
    SeedChunk c{};
    for (int j = 0; j < n; ++j) {
        const bnn_train_hparams& h = hp[(size_t)(s0 + j) * hp_stride];
        c.s[j] = SeedHp{h.lr, h.momentum, h.weight_decay, h.clip_norm, h.beta_in, h.beta_out, h.beta_in * (float)B,
                        h.beta_out * (float)B};
    }
    return c;
}

// The torch.optim.Adam scalars of one step, the bias corrections as torch computes them from Python floats (double),
// with this step's beta1
static AdamStep adam_step(const bnn_train_hparams& hp, const bnn_adam_hparams& adam) {
    const double t = (double)adam.step;
    AdamStep a;
    a.step_size = (float)((double)hp.lr / (1.0 - pow(adam.beta1, t)));
    a.bc2_sqrt = (float)sqrt(1.0 - pow(adam.beta2, t));
    a.w1 = (float)(1.0 - adam.beta1);
    a.beta2 = (float)adam.beta2;
    a.w2 = (float)(1.0 - adam.beta2);
    a.eps = (float)adam.eps;
    a.first = adam.step == 1;
    return a;
}

// One training step of n_seeds models, shared by the four entries: SGD (adam == null) or Adam.  Seed s's scalars are
// hp[s * hp_stride] (and adam[s * hp_stride]): stride 0 repeats one struct (bnn_train_step, bnn_train_step_adam),
// stride 1 reads one per seed (the _seeds entries); first_step and apply_update must be the same for every seed.  Every
// argument check runs before the device is touched.  Then the seed-group launches of the training kernel and, per chunk
// of SEED_CHUNK seeds, the fixed-order reduce, the logged metrics and the update.  `who` names the entry in messages;
// d_state0 / d_state1: the momentum buffer (SGD) or exp_avg / exp_avg_sq (Adam), required when apply_update.
// plan_seeds > 0: the seed groups and CTAs per seed are pick_plan's for plan_seeds seeds, whatever n_seeds is (0: for
// n_seeds); a seed's bits depend on its CTA count, so a fixed plan_seeds makes them independent of how many seeds share
// the call.  halt: the _halt entries, whose d_halted_at [n_seeds] (int64, 8-byte aligned) is required; the other entries
// pass null and the update kernels then compute what they did before the halt word existed.
static int train_step(const char* who, const bnn_model_config* cfg, const bnn_train_hparams* hp,
                      const bnn_adam_hparams* adam, bool is_adam, int hp_stride, int32_t n_seeds, int32_t plan_seeds,
                      bool halt, int64_t* d_halted_at, float* d_theta,
                      float* d_state0, float* d_state1, const float* d_x, const float* d_y, const int32_t* d_batch_index,
                      int64_t B, const float* d_eps_in, const float* d_eps12, const float* d_eps_sum, uint64_t seed,
                      uint64_t step, float* d_grad_out, float* d_metrics, void* d_workspace, cudaStream_t st) {
    BNN_REQUIRE(hp && (!is_adam || adam), BNN_E_ARG, "%s: null pointer", who);
    BNN_REQUIRE(n_seeds >= 1 && n_seeds <= 65535 && B >= 1 && B < (1ll << 30), BNN_E_ARG,
                "%s: n_seeds=%d B=%lld out of range", who, n_seeds, (long long)B);
    BNN_REQUIRE(plan_seeds >= 0 && plan_seeds <= 65535, BNN_E_ARG, "%s: plan_seeds=%d (0, or 1..65535)", who, plan_seeds);
    if (halt) {
        BNN_REQUIRE(d_halted_at, BNN_E_ARG, "%s: null d_halted_at", who);
        BNN_REQUIRE(step < (1ull << 63), BNN_E_ARG, "%s: step %llu does not fit the int64 halt word", who,
                    (unsigned long long)step);
        BNN_REQUIRE(((uintptr_t)d_halted_at & 7u) == 0, BNN_E_ALIGN, "%s: d_halted_at must be 8-byte aligned", who);
    }
    for (int s = 0; s < n_seeds; ++s) {
        const bnn_train_hparams& h = hp[(size_t)s * hp_stride];
        char at[32] = "";
        if (hp_stride) snprintf(at, sizeof(at), " (seed %d)", s);
        BNN_REQUIRE(h.first_step == hp[0].first_step && h.apply_update == hp[0].apply_update, BNN_E_ARG,
                    "%s: first_step and apply_update must be the same for every seed (seed %d differs from seed 0)", who, s);
        if (!is_adam) continue;
        // torch.optim.Adam's constructor checks, written so that NaN fails them too
        const bnn_adam_hparams& a = adam[(size_t)s * hp_stride];
        BNN_REQUIRE(h.lr >= 0.f, BNN_E_ARG, "%s: invalid learning rate %g%s", who, (double)h.lr, at);
        BNN_REQUIRE(h.weight_decay >= 0.f, BNN_E_ARG, "%s: invalid weight_decay %g%s", who, (double)h.weight_decay, at);
        BNN_REQUIRE(a.beta1 >= 0.0 && a.beta1 < 1.0, BNN_E_ARG, "%s: invalid beta1 %g (need [0, 1))%s", who, a.beta1, at);
        BNN_REQUIRE(a.beta2 >= 0.0 && a.beta2 < 1.0, BNN_E_ARG, "%s: invalid beta2 %g (need [0, 1))%s", who, a.beta2, at);
        BNN_REQUIRE(a.eps >= 0.0, BNN_E_ARG, "%s: invalid eps %g%s", who, a.eps, at);
        BNN_REQUIRE(a.step >= 1, BNN_E_ARG, "%s: step %lld (t is 1-based)%s", who, (long long)a.step, at);
    }
    const int first_step = hp[0].first_step, apply_update = hp[0].apply_update;
    int rc = validate_config(cfg);
    if (rc != BNN_OK) return rc;
    BNN_REQUIRE(d_theta && d_x && d_y && d_workspace, BNN_E_ARG, "%s: null pointer", who);
    BNN_REQUIRE(!apply_update || (d_state0 && (!is_adam || d_state1)), BNN_E_ARG, "%s: %s required to update", who,
                is_adam ? "exp_avg and exp_avg_sq" : "momentum buffer");
    const bool any = d_eps_in || d_eps12 || d_eps_sum, all = d_eps_in && d_eps12 && d_eps_sum;
    BNN_REQUIRE(!any || all, BNN_E_ARG, "%s: give all of eps_in, eps12, eps_sum or none", who);
    BNN_REQUIRE(aligned16(d_workspace) && (!d_eps12 || (aligned16(d_eps12) && aligned16(d_eps_sum))), BNN_E_ALIGN,
                "%s: workspace / eps12 / eps_sum must be 16-byte aligned", who);
    const int F = cfg->n_features, T = cfg->n_times, FP = (F + 3) & ~3;
    BNN_REQUIRE(shape_ok(cfg), BNN_E_CONFIG, "%s: compiled for the reference's shape T=100, F=41 (got T=%d, F=%d)", who, T, F);
    if ((rc = check_device()) != BNN_OK) return rc;
    const FlatLayout fl(F);
    const SeedPlan plan = pick_plan(cfg, B, plan_seeds ? plan_seeds : n_seeds);
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
    prm.saliency = 0; prm.gx_out = nullptr; prm.mu_out = nullptr;
    const bool tc = use_tc(cfg, B);
    const size_t smem = tc ? (size_t)tcx::SmemTC(cfg->zero_mask).total * sizeof(float) : (size_t)Smem3(T, F).total * sizeof(float);
    if (tc) {
        static PerDeviceOnce attr_tc_done;
        if (attr_tc_done.need()) {
            BNN_CUDA(cudaFuncSetAttribute(train_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        }
    } else {
        static PerDeviceOnce attr3_done;
        if (attr3_done.need()) {
            BNN_CUDA(cudaFuncSetAttribute(train_fwd_bwd3_kernel<100, 41>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          227 * 1024));
        }
    }
    // A group of more than TRAIN_SEED_CHUNK seeds runs one CTA per seed (pick_plan) and so more CTAs than SMs: it is
    // split into launches of a whole number of waves, which take as many waves in all as the group in one launch.
    const int sms = sm_count();
    const int sub = sms <= TRAIN_SEED_CHUNK ? TRAIN_SEED_CHUNK / sms * sms : TRAIN_SEED_CHUNK;
    for (int g0 = 0; g0 < n_seeds; g0 += plan.per) {   // seed groups (pick_plan); every buffer is indexed by the global seed
        const int g1 = n_seeds < g0 + plan.per ? n_seeds : g0 + plan.per;
        for (int s0 = g0; s0 < g1; s0 += sub) {
            const int n = g1 - s0 < sub ? g1 - s0 : sub;
            prm.seed0 = s0;
            for (int j = 0; j < n; ++j) prm.beta_out[j] = hp[(size_t)(s0 + j) * hp_stride].beta_out;
            if (tc) train_tc_kernel<<<dim3(n_cta, n), tcx::NTHR_TC, smem, st>>>(prm);
            else train_fwd_bwd3_kernel<100, 41><<<dim3(n_cta, n), NTHR3, smem, st>>>(prm);
        }
    }
    BNN_CUDA(cudaGetLastError());
    for (int s0 = 0; s0 < n_seeds; s0 += SEED_CHUNK) {   // seeds are independent from here on: chunk after chunk
        const int n = n_seeds - s0 < SEED_CHUNK ? n_seeds - s0 : SEED_CHUNK;
        const SeedChunk hc = seed_chunk(hp, hp_stride, s0, n, B);
        train_reduce_kernel<<<dim3(nb, n), 256, 0, st>>>(partial, d_theta, n_cta, fl.d, F, s0, hc, grad, sq);
        BNN_CUDA(cudaGetLastError());
        if (d_metrics) {
            train_metrics_kernel<<<n, 32, 0, st>>>(d_theta, grad, fl.d, F, (int)B, s0, hc, d_metrics);
            BNN_CUDA(cudaGetLastError());
        }
        if (is_adam) {
            AdamChunk ac{};
            for (int j = 0; j < n; ++j) ac.a[j] = adam_step(hp[(size_t)(s0 + j) * hp_stride], adam[(size_t)(s0 + j) * hp_stride]);
            train_adam_update_kernel<<<dim3(nb, n), 256, 0, st>>>(grad, sq, nb, fl.d, (int)B, s0, hc, ac, apply_update,
                                                                  d_theta, d_state0, d_state1, d_grad_out, d_metrics,
                                                                  d_halted_at, (int64_t)step);
        } else {
            train_update_kernel<<<dim3(nb, n), 256, 0, st>>>(grad, sq, nb, fl.d, (int)B, s0, hc, first_step, apply_update,
                                                             d_theta, d_state0, d_grad_out, d_metrics, d_halted_at,
                                                             (int64_t)step);
        }
        BNN_CUDA(cudaGetLastError());
    }
    return BNN_OK;
}

// The saliency launch of the v3 kernel (no input noise, no summary noise, upstream gradient (1, 0)) shared by
// bnn_saliency and bnn_posterior_saliency: n_models weight vectors [n_models, d] over B systems, grid (n_cta, n_models)
// with n_cta = SMs / n_models CTAs per model (one wave), at most one per pair of systems.  The caller has checked the
// arguments and the device.  Workspace: the CTAs' partials [n_models, n_cta, d + DPAD] (the saliency sums of squares
// sit in the dlv_in slot), then the producer warps' input-tile scratch.
static int64_t saliency_ctas(int32_t n_models, int64_t B) {
    int64_t n_cta = sm_count() / n_models;
    if (n_cta > (B + 1) / 2) n_cta = (B + 1) / 2;
    if (n_cta < 1) n_cta = 1;
    return n_cta;
}
// Sized for every call of at most n_models weight vectors and B systems, not just this one: n' * saliency_ctas(n', B')
// is not monotone (9 units over 31 systems run 144 CTAs, 10 run 140), so a walk that sizes its workspace for its full
// chunk and reuses it for a smaller remainder needs the bound.  n' * ctas <= max(n', SMs) (SMs / n' CTAs each up to SMs
// units, one each beyond) and <= n' * ceil(B' / 2), both non-decreasing in n' and B'.
static size_t saliency_workspace_floats(const bnn_model_config* cfg, int32_t n_models, int64_t B) {
    const int64_t sms = sm_count();
    int64_t n = n_models > sms ? n_models : sms;
    if (n > (int64_t)n_models * ((B + 1) / 2)) n = (int64_t)n_models * ((B + 1) / 2);
    return (size_t)n * (FlatLayout(cfg->n_features).d + DPAD) + 4 + (size_t)n * scratch_floats_per_cta(cfg);
}
static int saliency_launch(const bnn_model_config* cfg, int32_t n_models, const float* d_theta, const float* d_x, int64_t B,
                           const float* d_eps12, uint64_t seed, float* d_grad_x, float* d_mu, void* d_workspace,
                           cudaStream_t st, const float** partial_out, int* n_cta_out) {
    const int F = cfg->n_features, T = cfg->n_times;
    const FlatLayout fl(F);
    const int64_t n_cta = saliency_ctas(n_models, B);
    const int DP = fl.d + DPAD;
    float* partial = (float*)d_workspace;
    float* xprod = partial + (size_t)n_models * n_cta * DP;
    xprod += (4 - ((uintptr_t)xprod / sizeof(float)) % 4) % 4;
    Params prm;
    prm.theta = d_theta; prm.X = d_x; prm.Y = nullptr; prm.batch_index = nullptr;
    prm.eps_in = nullptr; prm.eps12 = d_eps12; prm.eps_sum = nullptr;
    prm.partial = partial; prm.head_rec = nullptr; prm.xprod = xprod;
    prm.B = (int)B; prm.T = T; prm.F = F; prm.FP = (F + 3) & ~3; prm.n_cta = (int)n_cta; prm.seed0 = 0;
    prm.seed = seed; prm.step = 0; prm.zero_mask = cfg->zero_mask;
    prm.hc = HeadConsts{cfg->lo_mu, cfg->hi_mu, cfg->lo_sd, cfg->hi_sd};
    prm.beta_out[0] = 0.f;   // every model reads entry 0 (train_v3.cuh)
    prm.saliency = 1; prm.gx_out = d_grad_x; prm.mu_out = d_mu;
    static PerDeviceOnce attr_done;
    if (attr_done.need()) {
        BNN_CUDA(cudaFuncSetAttribute(train_fwd_bwd3_kernel<100, 41>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      227 * 1024));
    }
    const size_t smem3 = (size_t)Smem3(T, F).total * sizeof(float);
    train_fwd_bwd3_kernel<100, 41><<<dim3((unsigned)n_cta, n_models), NTHR3, smem3, st>>>(prm);
    BNN_CUDA(cudaGetLastError());
    if (partial_out) *partial_out = partial;
    if (n_cta_out) *n_cta_out = (int)n_cta;
    return BNN_OK;
}

// ---- posterior attribution (bnn_posterior_saliency) ----
constexpr int ATTR_ROUNDS = S2 / 4;   // float4 blocks of eps1 | eps2 per (unit, row)

// eps12[u][r] = eps1 | eps2 of unit unit0 + u and row row0 + r, exactly the draws of the predictive kernel's Philox path
// (predict_tc.cuh, tail_draw_eps): block blk of counter (blk, global unit, global row, STREAM_EPS) under the raw seed.
__global__ void __launch_bounds__(256) attr_eps_kernel(int64_t n, int64_t rows, uint64_t seed, int64_t unit0, int64_t row0,
                                                       float* __restrict__ eps12) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    const int64_t ur = i / ATTR_ROUNDS;
    const int blk = (int)(i - ur * ATTR_ROUNDS);
    const int64_t u = ur / rows, r = ur - u * rows;
    reinterpret_cast<float4*>(eps12)[i] =
        philox_normal4(seed, STREAM_EPS, (uint32_t)(unit0 + u), (uint32_t)(row0 + r), (uint32_t)blk);
}

// One (unit, row, column) per thread: part[u][r] = (sum_t g[t][c]^2 for c < F | sum_t g[t][c] | mu) in double, t in
// increasing order.  A warp reads runs of consecutive columns of the same time step.
__global__ void __launch_bounds__(256) attr_unit_sums_kernel(const float* __restrict__ g, const float* __restrict__ mu,
                                                             int64_t n, int T, int F, double* __restrict__ part) {
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    const int64_t ur = i / F;
    const int c = (int)(i - ur * F);
    const float* p = g + ur * T * F + c;
    double s2 = 0.0, s1 = 0.0;
#pragma unroll 20
    for (int t = 0; t < T; ++t) {
        const double v = (double)__ldcs(p + (int64_t)t * F);
        s2 = fma(v, v, s2);
        s1 += v;
    }
    double* o = part + ur * (2 * F + 1);
    o[c] = s2;
    o[F + c] = s1;
    if (c == 0) o[2 * F] = (double)mu[ur];
}

// acc[r][j] (+)= part[u][r][j] for u = 0 .. n_units - 1 in that order (first: acc starts at part[0][r][j]); with
// finish_units > 0 the totals are divided in double and rounded once: attr[r][0][c] = acc / (U T), attr[r][1][c] = acc / U,
// mu_mean[r] = acc / U.  One thread per (row, accumulator); no atomics.
__global__ void __launch_bounds__(256) attr_accumulate_kernel(const double* __restrict__ part, int n_units, int64_t rows,
                                                              int T, int F, int first, int64_t finish_units,
                                                              double* __restrict__ acc, float* __restrict__ attr,
                                                              float* __restrict__ mu_mean) {
    const int W = 2 * F + 1;
    const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (i >= rows * W) return;
    const int64_t r = i / W;
    const int j = (int)(i - r * W);
    const int64_t ustride = rows * W;
    double a = first ? part[i] : acc[i] + part[i];
    for (int u = 1; u < n_units; ++u) a += part[u * ustride + i];
    acc[i] = a;
    if (finish_units > 0) {
        const double U = (double)finish_units;
        if (j < F) attr[r * 2 * F + j] = (float)(a / U / (double)T);
        else if (j < 2 * F) attr[r * 2 * F + j] = (float)(a / U);
        else mu_mean[r] = (float)(a / U);
    }
}

// workspace of one bnn_posterior_saliency call (floats, each block a multiple of 4): eps12 | g | mu | part | saliency
struct AttrWorkspace {
    size_t eps12, g, mu, part, sal, total;
    AttrWorkspace(const bnn_model_config* cfg, int32_t n_units, int64_t rows) {
        const size_t ur = (size_t)n_units * rows, F = cfg->n_features;
        size_t o = 0;
        eps12 = o; o += ur * S2;
        g = o; o += ur * cfg->n_times * F;
        mu = o; o += (ur + 3) & ~(size_t)3;
        part = o; o += (ur * (2 * F + 1) * 2 + 3) & ~(size_t)3;
        sal = o; o += saliency_workspace_floats(cfg, n_units, rows);
        total = o;
    }
};

}  // namespace train
}  // namespace bnn

extern "C" {

size_t bnn_train_workspace_bytes(const bnn_model_config* cfg, int64_t B, int32_t n_seeds) {
    using namespace bnn;
    if (validate_config(cfg) != BNN_OK || B <= 0 || n_seeds <= 0) return 0;
    return train::workspace_bytes(cfg, B, n_seeds, train::pick_plan(cfg, B, n_seeds).n_cta);
}

size_t bnn_train_workspace_bytes_seeds(const bnn_model_config* cfg, int64_t B, int32_t n_seeds, int32_t plan_seeds) {
    using namespace bnn;
    if (validate_config(cfg) != BNN_OK || B <= 0 || n_seeds <= 0 || plan_seeds < 0 || plan_seeds > 65535) return 0;
    return train::workspace_bytes(cfg, B, n_seeds, train::pick_plan(cfg, B, plan_seeds ? plan_seeds : n_seeds).n_cta);
}

int bnn_train_step(const bnn_model_config* cfg, const bnn_train_hparams* hp, int32_t n_seeds, float* d_theta,
                   float* d_momentum, const float* d_x, const float* d_y, const int32_t* d_batch_index, int64_t B,
                   const float* d_eps_in, const float* d_eps12, const float* d_eps_sum, uint64_t seed, uint64_t step,
                   float* d_grad_out, float* d_metrics, void* d_workspace, void* stream) {
    return bnn::train::train_step("bnn_train_step", cfg, hp, nullptr, false, 0, n_seeds, 0, false, nullptr, d_theta,
                                  d_momentum, nullptr, d_x,
                                  d_y, d_batch_index, B, d_eps_in, d_eps12, d_eps_sum, seed, step, d_grad_out, d_metrics,
                                  d_workspace, (cudaStream_t)stream);
}

int bnn_train_step_seeds(const bnn_model_config* cfg, const bnn_train_hparams* hp, int32_t n_seeds, int32_t plan_seeds,
                         float* d_theta, float* d_momentum, const float* d_x, const float* d_y, const int32_t* d_batch_index, int64_t B,
                         const float* d_eps_in, const float* d_eps12, const float* d_eps_sum, uint64_t seed, uint64_t step,
                         float* d_grad_out, float* d_metrics, void* d_workspace, void* stream) {
    return bnn::train::train_step("bnn_train_step_seeds", cfg, hp, nullptr, false, 1, n_seeds, plan_seeds, false, nullptr,
                                  d_theta, d_momentum, nullptr,
                                  d_x, d_y, d_batch_index, B, d_eps_in, d_eps12, d_eps_sum, seed, step, d_grad_out,
                                  d_metrics, d_workspace, (cudaStream_t)stream);
}

int bnn_train_step_adam(const bnn_model_config* cfg, const bnn_train_hparams* hp, const bnn_adam_hparams* adam,
                        int32_t n_seeds, float* d_theta, float* d_exp_avg, float* d_exp_avg_sq, const float* d_x,
                        const float* d_y, const int32_t* d_batch_index, int64_t B, const float* d_eps_in,
                        const float* d_eps12, const float* d_eps_sum, uint64_t seed, uint64_t step, float* d_grad_out,
                        float* d_metrics, void* d_workspace, void* stream) {
    return bnn::train::train_step("bnn_train_step_adam", cfg, hp, adam, true, 0, n_seeds, 0, false, nullptr, d_theta,
                                  d_exp_avg, d_exp_avg_sq,
                                  d_x, d_y, d_batch_index, B, d_eps_in, d_eps12, d_eps_sum, seed, step, d_grad_out,
                                  d_metrics, d_workspace, (cudaStream_t)stream);
}

int bnn_train_step_adam_seeds(const bnn_model_config* cfg, const bnn_train_hparams* hp, const bnn_adam_hparams* adam,
                              int32_t n_seeds, int32_t plan_seeds, float* d_theta, float* d_exp_avg, float* d_exp_avg_sq, const float* d_x,
                              const float* d_y, const int32_t* d_batch_index, int64_t B, const float* d_eps_in,
                              const float* d_eps12, const float* d_eps_sum, uint64_t seed, uint64_t step, float* d_grad_out,
                              float* d_metrics, void* d_workspace, void* stream) {
    return bnn::train::train_step("bnn_train_step_adam_seeds", cfg, hp, adam, true, 1, n_seeds, plan_seeds, false, nullptr,
                                  d_theta, d_exp_avg,
                                  d_exp_avg_sq, d_x, d_y, d_batch_index, B, d_eps_in, d_eps12, d_eps_sum, seed, step,
                                  d_grad_out, d_metrics, d_workspace, (cudaStream_t)stream);
}

int bnn_train_step_seeds_halt(const bnn_model_config* cfg, const bnn_train_hparams* hp, int32_t n_seeds, int32_t plan_seeds,
                              float* d_theta, float* d_momentum, const float* d_x, const float* d_y,
                              const int32_t* d_batch_index, int64_t B, const float* d_eps_in, const float* d_eps12,
                              const float* d_eps_sum, uint64_t seed, uint64_t step, float* d_grad_out, float* d_metrics,
                              void* d_workspace, int64_t* d_halted_at, void* stream) {
    return bnn::train::train_step("bnn_train_step_seeds_halt", cfg, hp, nullptr, false, 1, n_seeds, plan_seeds, true,
                                  d_halted_at, d_theta, d_momentum, nullptr, d_x, d_y, d_batch_index, B, d_eps_in, d_eps12,
                                  d_eps_sum, seed, step, d_grad_out, d_metrics, d_workspace, (cudaStream_t)stream);
}

int bnn_train_step_adam_seeds_halt(const bnn_model_config* cfg, const bnn_train_hparams* hp, const bnn_adam_hparams* adam,
                                   int32_t n_seeds, int32_t plan_seeds, float* d_theta, float* d_exp_avg,
                                   float* d_exp_avg_sq, const float* d_x, const float* d_y, const int32_t* d_batch_index,
                                   int64_t B, const float* d_eps_in, const float* d_eps12, const float* d_eps_sum,
                                   uint64_t seed, uint64_t step, float* d_grad_out, float* d_metrics, void* d_workspace,
                                   int64_t* d_halted_at, void* stream) {
    return bnn::train::train_step("bnn_train_step_adam_seeds_halt", cfg, hp, adam, true, 1, n_seeds, plan_seeds, true,
                                  d_halted_at, d_theta, d_exp_avg, d_exp_avg_sq, d_x, d_y, d_batch_index, B, d_eps_in,
                                  d_eps12, d_eps_sum, seed, step, d_grad_out, d_metrics, d_workspace, (cudaStream_t)stream);
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
    cudaStream_t st = (cudaStream_t)stream;
    const float* partial = nullptr;
    int n_cta = 0;
    rc = train::saliency_launch(cfg, n_models, d_theta, d_x, B, d_eps12, seed, d_grad_x, d_mu, d_workspace, st, &partial,
                                &n_cta);
    if (rc != BNN_OK) return rc;
    train::saliency_finish_kernel<<<n_models, 64, 0, st>>>(partial, n_cta, FlatLayout(cfg->n_features).d, cfg->n_features,
                                                           d_sumsq);
    BNN_CUDA(cudaGetLastError());
    return BNN_OK;
}

size_t bnn_posterior_saliency_workspace_bytes(const bnn_model_config* cfg, int32_t n_units, int64_t rows) {
    using namespace bnn;
    if (validate_config(cfg) != BNN_OK || n_units < 1 || n_units > 65535 || rows < 1 || rows >= (1ll << 30)) return 0;
    return train::AttrWorkspace(cfg, n_units, rows).total * sizeof(float);
}

int bnn_posterior_saliency(const bnn_model_config* cfg, int32_t n_units, const float* d_theta, int64_t unit0,
                           const float* d_x, int64_t rows, int64_t row0, uint64_t seed, double* d_acc, int32_t first,
                           int64_t finish_units, float* d_attr, float* d_mu_mean, float* d_mu_units, void* d_workspace,
                           void* stream) {
    using namespace bnn;
    int rc = validate_config(cfg);
    if (rc != BNN_OK) return rc;
    const char* who = "bnn_posterior_saliency";
    BNN_REQUIRE(d_theta && d_x && d_acc && d_workspace, BNN_E_ARG, "%s: null pointer", who);
    BNN_REQUIRE(finish_units == 0 || (d_attr && d_mu_mean), BNN_E_ARG, "%s: finishing needs d_attr and d_mu_mean", who);
    BNN_REQUIRE(n_units >= 1 && n_units <= 65535 && rows >= 1 && rows < (1ll << 30), BNN_E_ARG,
                "%s: n_units=%d rows=%lld out of range", who, n_units, (long long)rows);
    BNN_REQUIRE(unit0 >= 0 && unit0 + n_units <= (1ll << 32) && row0 >= 0 && row0 + rows <= (1ll << 32), BNN_E_ARG,
                "%s: unit0=%lld row0=%lld: global unit and row indices must fit the 32-bit Philox counters", who,
                (long long)unit0, (long long)row0);
    BNN_REQUIRE(finish_units == 0 || (finish_units >= n_units && finish_units < (1ll << 32)), BNN_E_ARG,
                "%s: finish_units=%lld (0, or the number of units accumulated, >= n_units)", who, (long long)finish_units);
    BNN_REQUIRE(cfg->n_times == 100 && cfg->n_features == 41, BNN_E_CONFIG,
                "%s: compiled for T=100, F=41 (got T=%d, F=%d)", who, cfg->n_times, cfg->n_features);
    BNN_REQUIRE(aligned16(d_workspace) && ((uintptr_t)d_acc & 7u) == 0 && ((uintptr_t)d_x & 3u) == 0 &&
                    ((uintptr_t)d_theta & 3u) == 0 && ((uintptr_t)d_attr & 3u) == 0 && ((uintptr_t)d_mu_mean & 3u) == 0 &&
                    ((uintptr_t)d_mu_units & 3u) == 0,
                BNN_E_ALIGN, "%s: d_workspace must be 16-byte, d_acc 8-byte and the float arrays 4-byte aligned", who);
    if ((rc = check_device()) != BNN_OK) return rc;
    const int F = cfg->n_features, T = cfg->n_times;
    const train::AttrWorkspace wl(cfg, n_units, rows);
    float* ws = (float*)d_workspace;
    float* eps12 = ws + wl.eps12;
    float* g = ws + wl.g;
    float* mu = d_mu_units ? d_mu_units : ws + wl.mu;
    double* part = reinterpret_cast<double*>(ws + wl.part);
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t ur = (int64_t)n_units * rows;
    const int64_t n_eps = ur * train::ATTR_ROUNDS, n_sums = ur * F, n_acc = rows * (2 * F + 1);
    train::attr_eps_kernel<<<(unsigned)((n_eps + 255) / 256), 256, 0, st>>>(n_eps, rows, seed, unit0, row0, eps12);
    BNN_CUDA(cudaGetLastError());
    rc = train::saliency_launch(cfg, n_units, d_theta, d_x, rows, eps12, seed, g, mu, ws + wl.sal, st, nullptr, nullptr);
    if (rc != BNN_OK) return rc;
    train::attr_unit_sums_kernel<<<(unsigned)((n_sums + 255) / 256), 256, 0, st>>>(g, mu, n_sums, T, F, part);
    BNN_CUDA(cudaGetLastError());
    train::attr_accumulate_kernel<<<(unsigned)((n_acc + 255) / 256), 256, 0, st>>>(part, n_units, rows, T, F, first ? 1 : 0,
                                                                                   finish_units, d_acc, d_attr, d_mu_mean);
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

/*
 * bnnchaos.h -- C ABI of libbnnchaos.so: the B200 (sm_100a) kernels behind the drop-in
 * replacement of bnn_chaos_model's MultiSWAG posterior-predictive and SWAG-training path.
 *
 * The reference has no FFI: the path sits behind a Python class API
 * (/root/reference/spock_reg_model.py:339-967, VarModel / SWAGModel / save_swag /
 * load_swag).  Each entry point below names the reference method(s) it replaces; the
 * Python host mirror (bnn_chaos_model_b200/spock_reg_model.py) binds them with ctypes --
 * see INTEGRATION.md for the stub a maintainer of the reference would add.
 *
 * Conventions
 *   - every pointer named d_* is a DEVICE pointer to contiguous fp32 (or int32 where said),
 *     16-byte aligned, owned by the caller; h_* are HOST pointers;
 *   - `stream` is a cudaStream_t passed as void*; the library only enqueues work on it and
 *     never synchronises (except the h_* convenience entry points, which say so);
 *   - return value: 0 ok; >0 a cudaError_t; <0 an argument error (BNN_E_*);
 *     bnn_last_error_string() describes the last failure on the calling thread;
 *   - no allocation, no global mutable state except one-time cudaFuncSetAttribute;
 *   - sm_100a only: every entry point returns BNN_E_ARCH on another device.  There is no
 *     CPU fallback.
 */
#ifndef BNNCHAOS_H_
#define BNNCHAOS_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BNN_ABI_VERSION 1

enum {
    BNN_OK = 0,
    BNN_E_ARG = -1,     /* null pointer / bad size */
    BNN_E_CONFIG = -2,  /* model shape not supported by the compiled kernels */
    BNN_E_ARCH = -3,    /* device is not sm_100 */
    BNN_E_ALIGN = -4    /* pointer not 16-byte aligned */
};

/* Model description: VarModel.__init__ (spock_reg_model.py:341-402). */
typedef struct bnn_model_config {
    int32_t n_features;   /* F: hparams['time_series_features'] (41)              :348-358 */
    int32_t hidden;       /* H: hparams['hidden'] (40)                            :359-360 */
    int32_t latent;       /* L: hparams['latent'] (20)                            :359-362 */
    int32_t n_in_layers;  /* hparams['in']  (1): hidden->hidden layers, feature_nn :359   */
    int32_t n_out_layers; /* hparams['out'] (1): hidden->hidden layers, regress_nn :360   */
    int32_t n_times;      /* T: time steps per system (100); runtime, 4 <= T, T % 4 == 0   */
    uint64_t zero_mask;   /* bit c set <=> column c is zeroed by zero_megno/mmr/nan/
                             eplusminus (:452-478) under this model's include_* flags      */
    float lo_mu, hi_mu;   /* soft_clamp bounds of mu  (4, 12)                     :440     */
    float lo_sd, hi_sd;   /* soft_clamp bounds of std (self.lowest = 0.5|0.1, 6)  :441     */
} bnn_model_config;

int bnn_abi_version(void);
const char* bnn_last_error_string(void);

/* d: length of SWAGModel.flatten() (:734-746) for this config, or <0. */
int64_t bnn_param_count(const bnn_model_config* cfg);
/* P: floats per unit of the kernel-side ("packed") weight layout, or <0. */
int64_t bnn_packed_param_count(const bnn_model_config* cfg);

/* ---------------------------------------------------------------------------------------
 * SWAGModel.sample_weights (:815-838) for U = n_units (model, weight-sample) units at once:
 *   theta = w_avg + (scale/sqrt2 * z1) * sqrt|w2_avg - w_avg^2| + scale * (D z2) / sqrt(2(K-1)),
 *   D = pre_D - w_avg[:,None].
 * Unit u uses model d_unit_model[u] (NULL: model = (unit_offset+u) / samples_per_model).
 * d_z1 [U,d] / d_z2 [U,K] explicit normal draws (the reference's randn((1,d)), randn((K,1))),
 * or both NULL: drawn in-kernel from Philox4x32-10 keyed on (seed; unit_offset+u, element).
 * Outputs (either may be NULL, not both): d_theta [U,d] in flatten() order (what SWAGModel.load()
 * would install, :748-761) and d_theta_packed [U,P] in the layout bnn_predict consumes.  One fused
 * launch: the packed layout is written from shared memory, theta never round-trips through HBM.
 * pre_D is [M,d,K] row-major, exactly the saved tensor (:917).
 */
int bnn_swag_sample(const bnn_model_config* cfg, const float* d_w_avg, const float* d_w2_avg,
                    const float* d_pre_D, int32_t n_models, int32_t K, const int32_t* d_unit_model,
                    int64_t n_units, int64_t unit_offset, int32_t samples_per_model, float scale,
                    uint64_t seed, const float* d_z1, const float* d_z2, float* d_theta,
                    float* d_theta_packed, void* stream);

/* SWAGModel.load (:748-761) for the kernels: flatten()-order theta [U,d] -> packed [U,P]. */
int bnn_pack_theta(const bnn_model_config* cfg, const float* d_theta, int64_t n_units,
                   float* d_theta_packed, void* stream);

/* ---------------------------------------------------------------------------------------
 * SWAGModel.forward_swag_fast / forward_swag (:840-908) and VarModel.forward(noisy_val=False)
 * (:486-528) for every (unit, system) pair in one launch:
 *   zero_* masks -> feature_nn per time step -> mean / unbiased variance over time ->
 *   sampled summary statistics (eps1, eps2) -> regress_nn -> soft_clamp.
 * d_x [N,T,F] already StandardScaler-normalised (as every reference caller passes it).
 * d_eps [U,N,2L] explicit draws (eps1 = [..., :L], eps2 = [..., L:], the two randn_like of
 * :426-427), or NULL: Philox keyed on (seed; unit_offset+u, system_offset+n, element).
 * d_eps_sum [U,N,2L] or NULL: add_summary_noise (:448-450, VarModel.forward(noisy_val=True));
 * the input noise of that path (:444-446) is applied beforehand by bnn_add_input_noise.
 * d_out [U,N,2] (mu, std) when out_system_major == 0, else [N,U,2].
 * d_summary_out [U,N,2L] or NULL: the summary statistics compute_summary_stats returns
 * (:416-435), before any summary noise -- what _summary_kl is computed from (:515-520).
 * d_workspace: bnn_predict_workspace_bytes() bytes (may be NULL when that returns 0).
 */
size_t bnn_predict_workspace_bytes(const bnn_model_config* cfg, int64_t n_systems, int64_t n_units);
/* Systems per position-independent group of the kernel bnn_predict selects for cfg (or <0): a batch split at
 * multiples of it (shards, chunks) gives bit-identical per-system results to the unsplit batch.  The FFMA
 * kernels treat every system alike (1); the tensor-core kernel pools in 32-row blocks of its 5-system tile (5). */
int32_t bnn_predict_system_granule(const bnn_model_config* cfg);
int bnn_predict(const bnn_model_config* cfg, const float* d_x, int64_t n_systems,
                const float* d_theta_packed, int64_t n_units, const float* d_eps,
                const float* d_eps_sum, uint64_t seed, int64_t unit_offset, int64_t system_offset,
                int32_t out_system_major, float* d_out, float* d_summary_out, void* d_workspace,
                void* stream);
/* The same with explicit output strides (in floats, even): the (mu, std) pair of (unit u, system n) of THIS call goes to
 * d_out + u * out_unit_stride + n * out_system_stride.  Lets a caller fill a column block of a larger [N, U_total, 2]
 * array from one chunk of units (weights sampled chunk by chunk: 60,000 units x 77 kB never exist at once). */
int bnn_predict_strided(const bnn_model_config* cfg, const float* d_x, int64_t n_systems,
                        const float* d_theta_packed, int64_t n_units, const float* d_eps,
                        const float* d_eps_sum, uint64_t seed, int64_t unit_offset, int64_t system_offset,
                        int64_t out_unit_stride, int64_t out_system_stride, float* d_out,
                        float* d_summary_out, void* d_workspace, void* stream);

/* VarModel.add_input_noise (:444-446) after the zero_* masks (:487-500):
 * x_noisy = x (zeroed columns set to 0) + eps_in * exp(input_noise_logvar/2).
 * d_x, d_eps_in, d_x_noisy [n_rows = B*T, F]; d_lv_in [F].  The result is then passed to
 * bnn_predict with a config whose zero_mask is 0 (every column carries noise). */
int bnn_add_input_noise(const bnn_model_config* cfg, const float* d_x, const float* d_eps_in,
                        const float* d_lv_in, int64_t n_rows, float* d_x_noisy, void* stream);

/* VarModel.predict_instability (:437-442): regress_nn + soft_clamp on given summary
 * statistics d_summary [B,2L] with ONE unit of packed weights -> d_out [B,2]. */
int bnn_predict_instability(const bnn_model_config* cfg, const float* d_summary, int64_t B,
                            const float* d_theta_packed, float* d_out, void* stream);

/* Host-buffer convenience entry (what a non-torch caller binds): h_x [N,T,F] and h_out [U,N,2]
 * are HOST buffers (pinned for real overlap); SWAG statistics are device-resident.  Samples U =
 * n_models*samples_per_model units with Philox and predicts; the systems are cut into up to four
 * chunks (at multiples of bnn_predict_system_granule) whose upload / prediction / download are
 * pipelined over two internal side streams; synchronises before returning.  Bit-identical to one
 * bnn_swag_sample + bnn_predict on device-resident data.
 * d_scratch must hold bnn_multiswag_host_scratch_bytes() bytes of device memory. */
size_t bnn_multiswag_host_scratch_bytes(const bnn_model_config* cfg, int64_t n_systems, int64_t n_units);
int bnn_multiswag_predict_host(const bnn_model_config* cfg, const float* h_x, int64_t n_systems,
                               const float* d_w_avg, const float* d_w2_avg, const float* d_pre_D,
                               int32_t n_models, int32_t K, int32_t samples_per_model, float scale,
                               uint64_t seed, float* h_out, void* d_scratch, void* stream);

/* ---------------------------------------------------------------------------------------
 * VarModel._lossfnc (:547-577) + safe_log_erf (:323-335), forward and analytic backward:
 * d_mu_sd [B,2], d_y [B,2] -> d_loss_per_system [B] (may be NULL), d_loss_sum [1] (may be
 * NULL; accumulated deterministically), d_grad [B,2] = d(sum loss)/d(mu,sd) (may be NULL).
 */
int bnn_nll_fwd_bwd(const float* d_mu_sd, const float* d_y, int64_t B, float* d_loss_per_system,
                    float* d_loss_sum, float* d_grad, void* stream);

/* ---------------------------------------------------------------------------------------
 * SWAGModel.training_step (:722-732) + loss.backward() + clip_grad_norm_ + torch.optim.SGD
 * (:709-711; run_swag.py:61,74-79) for n_seeds independent models in one call:
 *   total = sum_b _lossfnc(forward(x_b, noisy_val=True), y_b) + input_kl*beta_in*B + summary_kl*beta_out
 *   g = d total / d theta (analytic);  g *= min(1, clip/(|g|_2 + 1e-6));  d_p = g + wd*theta;
 *   buf = d_p (first step) | momentum*buf + d_p;  theta -= lr*buf.
 * State per seed (device, caller-owned): d_theta [n_seeds,d] in flatten() order, d_momentum [n_seeds,d].
 * d_x [n_data,T,F] normalised inputs, d_y [n_data,2]; seed s's batch row b is data row
 * d_batch_index[s*B+b] (int32; NULL: row b, every seed sees the same batch).  The zero_* masks of cfg are
 * applied before the input noise, like forward() (:487-506).
 * Noise: explicit d_eps_in [n_seeds,B,T,F], d_eps12 [n_seeds,B,2L] (eps1 | eps2 of :426-427), d_eps_sum
 * [n_seeds,B,2L] (the randn_like draws of :445, :426-427, :449), or all NULL: Philox4x32-10 keyed on
 * (seed; seed index, batch position, step) -- bnn_train_noise writes exactly those draws out.
 * d_grad_out [n_seeds,d] (may be NULL): the gradient before clipping.
 * d_metrics [n_seeds,8] (may be NULL): train_loss_no_reg, train_loss_with_reg, input_kl, summary_kl (each
 * / B, as logged :731), grad norm, clip coefficient (<= 1), non-finite flag (terminate_on_nan,
 * run_swag.py:78, without a host sync), reserved.
 * d_workspace: bnn_train_workspace_bytes() bytes, 16-byte aligned.  Gradient partials are reduced in a
 * fixed order: the step is bit-reproducible.  T/4 * ceil(F/4) <= 288 and F <= 48 (else BNN_E_CONFIG).
 */
typedef struct bnn_train_hparams {
    float lr, momentum, weight_decay, clip_norm; /* swa_lr, 0.9, hparams.weight_decay, 0.1*d */
    float beta_in, beta_out;                     /* find_minima.py:50-51                     */
    int32_t first_step;                          /* 1: momentum buffer is initialised (SGD)  */
    int32_t apply_update;                        /* 0: gradients / metrics only              */
} bnn_train_hparams;

size_t bnn_train_workspace_bytes(const bnn_model_config* cfg, int64_t B, int32_t n_seeds);
int bnn_train_step(const bnn_model_config* cfg, const bnn_train_hparams* hp, int32_t n_seeds,
                   float* d_theta, float* d_momentum, const float* d_x, const float* d_y,
                   const int32_t* d_batch_index, int64_t B, const float* d_eps_in,
                   const float* d_eps12, const float* d_eps_sum, uint64_t seed, uint64_t step,
                   float* d_grad_out, float* d_metrics, void* d_workspace, void* stream);

/* The same step with torch.optim.Adam (amsgrad=False, maximize=False) in place of SGD -- what a caller of
 * clip_grad_norm_ + Adam.step() after the training step's backward gets.  Weight decay is L2 added to the gradient
 * (not AdamW):
 *   g *= min(1, clip/(|g|_2 + 1e-6));  g += wd*theta;  m = m + (1-beta1)(g - m);  v = beta2 v + (1-beta2) g^2;
 *   theta -= lr/(1 - beta1^t) * m / (sqrt(v)/sqrt(1 - beta2^t) + eps).
 * The bias corrections are computed in double from this call's beta1 / beta2 / t, as torch does; beta1 may change from
 * call to call (the one-cycle schedule sets betas[0] every step).  At t == 1 d_exp_avg / d_exp_avg_sq are not read (a
 * fresh optimizer's zero state): they need no initialisation.
 * From hp: lr, weight_decay, clip_norm, beta_in, beta_out, apply_update; momentum and first_step are not read.
 * State per seed (device, caller-owned): d_exp_avg, d_exp_avg_sq [n_seeds,d] (required when apply_update = 1;
 * apply_update = 0 leaves theta and both buffers untouched).  BNN_E_ARG for what torch.optim.Adam rejects: lr < 0,
 * weight_decay < 0, beta outside [0, 1), eps < 0, and t < 1.  Every other argument, the metrics and the workspace
 * (bnn_train_workspace_bytes) as bnn_train_step.
 */
typedef struct bnn_adam_hparams {
    double beta1, beta2, eps;  /* torch.optim.Adam betas / eps; beta1 may change per call (one-cycle schedule) */
    int64_t step;              /* t of this update, 1-based; t == 1: both moment buffers are treated as zero */
} bnn_adam_hparams;

int bnn_train_step_adam(const bnn_model_config* cfg, const bnn_train_hparams* hp, const bnn_adam_hparams* adam,
                        int32_t n_seeds, float* d_theta, float* d_exp_avg, float* d_exp_avg_sq, const float* d_x,
                        const float* d_y, const int32_t* d_batch_index, int64_t B, const float* d_eps_in,
                        const float* d_eps12, const float* d_eps_sum, uint64_t seed, uint64_t step,
                        float* d_grad_out, float* d_metrics, void* d_workspace, void* stream);

/* Per-seed hyperparameters (hyperparameter sweeps in one fused job): bnn_train_step / bnn_train_step_adam with HOST
 * arrays hp [n_seeds] (and adam [n_seeds]).  Seed s uses hp[s] for lr, momentum, weight_decay, clip_norm, beta_in and
 * beta_out -- in the summary-KL term of its gradient, its KL scales, its clip, its update and its logged metrics -- and
 * adam[s] for beta1, beta2, eps and t (bias corrections in double per seed, as bnn_train_step_adam computes them).
 * first_step and apply_update must be equal across seeds.  The values travel in the kernels' parameters: no allocation,
 * no copy, no synchronisation.  With all entries equal the results are those of the single-struct entry bit for bit, and
 * seed s's results are those of a call in which every seed carries hp[s] (same plan, same Philox key).  Every other
 * argument and the workspace (bnn_train_workspace_bytes) as the single-struct entry.  BNN_E_ARG: a null hp / adam, mixed
 * first_step or apply_update, and (Adam) a seed's lr < 0, weight_decay < 0, beta outside [0, 1), eps < 0 or t < 1, the
 * message naming the seed; every check runs before the device is touched.
 * plan_seeds: 0 plans the seed groups and the CTAs per seed for n_seeds, as the single-struct entry does; > 0 plans them
 * for plan_seeds seeds whatever n_seeds is (n_seeds seeds run in groups of that plan's size, each seed on that plan's
 * CTAs).  A seed's bits depend on its CTA count, so a fixed plan_seeds gives a seed the same result whichever and
 * however many seeds share the call: a job split over any number of GPUs trains each run identically.  The workspace is
 * bnn_train_workspace_bytes_seeds(cfg, B, n_seeds, plan_seeds) bytes (plan_seeds = 0: bnn_train_workspace_bytes). */
size_t bnn_train_workspace_bytes_seeds(const bnn_model_config* cfg, int64_t B, int32_t n_seeds, int32_t plan_seeds);
int bnn_train_step_seeds(const bnn_model_config* cfg, const bnn_train_hparams* hp, int32_t n_seeds, int32_t plan_seeds,
                         float* d_theta, float* d_momentum, const float* d_x, const float* d_y,
                         const int32_t* d_batch_index, int64_t B, const float* d_eps_in,
                         const float* d_eps12, const float* d_eps_sum, uint64_t seed, uint64_t step,
                         float* d_grad_out, float* d_metrics, void* d_workspace, void* stream);
int bnn_train_step_adam_seeds(const bnn_model_config* cfg, const bnn_train_hparams* hp, const bnn_adam_hparams* adam,
                              int32_t n_seeds, int32_t plan_seeds, float* d_theta, float* d_exp_avg, float* d_exp_avg_sq, const float* d_x,
                              const float* d_y, const int32_t* d_batch_index, int64_t B, const float* d_eps_in,
                              const float* d_eps12, const float* d_eps_sum, uint64_t seed, uint64_t step,
                              float* d_grad_out, float* d_metrics, void* d_workspace, void* stream);
/* Per-seed halt on a non-finite step: bnn_train_step_seeds / bnn_train_step_adam_seeds plus d_halted_at [n_seeds], a
 * caller-owned device int64 per seed: -1 while the seed's run is live, else the `step` argument of the call at which it
 * halted.  Step k is bad for seed s when nll + skl + norm is not finite -- the batch NLL sum, the summary-KL term times
 * beta_out and the L2 norm of the unclipped gradient, the condition of metrics column 6 (input-KL overflow reaches it
 * through its gradient).  When seed s is already halted, or step k is bad for it, the update of s is not applied: theta,
 * the momentum buffer and exp_avg / exp_avg_sq of s stay bit for bit what they were before the call; a live seed
 * latches d_halted_at[s] = k.  So the offending step is not applied.  (Whether the reference's terminate_on_nan checked
 * before or after optimizer.step() is unverified: its Lightning 1.1 source is not available.)  d_grad_out and d_metrics
 * are written for every seed as by the _seeds entry, and a halted seed's forward / backward still runs.  Seeds are
 * independent: a live seed's bits do not depend on whether another seed halted, and with every word -1 and no bad step
 * the results are the _seeds entry's bit for bit.  The decision is made on the device at the step itself; the caller
 * reads the words whenever it synchronises anyway.  The _seeds entries are these with no halt word.  BNN_E_ARG: a null
 * d_halted_at, a step >= 2^63 (it must fit the word); BNN_E_ALIGN: d_halted_at not 8-byte aligned; both come back
 * before the device is touched, with the _seeds entry's own checks. */
int bnn_train_step_seeds_halt(const bnn_model_config* cfg, const bnn_train_hparams* hp, int32_t n_seeds, int32_t plan_seeds,
                              float* d_theta, float* d_momentum, const float* d_x, const float* d_y,
                              const int32_t* d_batch_index, int64_t B, const float* d_eps_in, const float* d_eps12,
                              const float* d_eps_sum, uint64_t seed, uint64_t step, float* d_grad_out, float* d_metrics,
                              void* d_workspace, int64_t* d_halted_at, void* stream);
int bnn_train_step_adam_seeds_halt(const bnn_model_config* cfg, const bnn_train_hparams* hp, const bnn_adam_hparams* adam,
                                   int32_t n_seeds, int32_t plan_seeds, float* d_theta, float* d_exp_avg,
                                   float* d_exp_avg_sq, const float* d_x, const float* d_y, const int32_t* d_batch_index,
                                   int64_t B, const float* d_eps_in, const float* d_eps12, const float* d_eps_sum,
                                   uint64_t seed, uint64_t step, float* d_grad_out, float* d_metrics, void* d_workspace,
                                   int64_t* d_halted_at, void* stream);
/* Saliency (figures/feature_importance.py:93-131, gradforward): for each of n_models weight vectors d_theta[m]
 * (flatten() order; the script uses w_avg) and each system b: mu_b = predict_instability(compute_summary_stats(
 * mask(x_b)))[0] and g = d mu_b / d x (all F columns of the masked input; no input noise, no summary noise).
 * eps1 | eps2 of compute_summary_stats (:426-427): explicit d_eps12 [n_models,B,2L] or NULL (Philox on (seed; model,
 * system)).  Outputs: d_grad_x [n_models,B,T,F] (may be NULL), d_sumsq [n_models,F] = sum over systems and time steps
 * of g^2 (the script's importance is this / (B*T)), d_mu [n_models,B].  Workspace: bnn_train_workspace_bytes(cfg, B,
 * n_models).  T = 100, F = 41 only (else BNN_E_CONFIG). */
int bnn_saliency(const bnn_model_config* cfg, int32_t n_models, const float* d_theta, const float* d_x, int64_t B,
                 const float* d_eps12, uint64_t seed, float* d_grad_x, float* d_sumsq, float* d_mu, void* d_workspace,
                 void* stream);

/* Posterior attribution: which inputs drive each row's predicted mean under the MultiSWAG posterior.  For the n_units
 * sampled weight vectors d_theta [n_units, d] (flatten() order; global units unit0 ..) and the model-input rows d_x
 * [rows, T, F] (global rows row0 ..): mu_u is unit u's predicted mean with the predictive kernel's own summary draws
 * (eps1 | eps2 = Philox on (seed; unit0 + u, row0 + r), exactly bnn_predict's with d_eps NULL) and no input or summary
 * noise, and g_u = d mu_u / d x_r [T, F] (the saliency kernel of bnn_saliency; the zeroed columns carry gradient too).
 * Per row, into the caller's double accumulators d_acc [rows, 2F + 1]:
 *   acc[r][c] += sum_t g_u[t][c]^2,  acc[r][F + c] += sum_t g_u[t][c],  acc[r][2F] += mu_u,
 * unit after unit in increasing order (first != 0: the accumulators start at this call's first unit, unread), each
 * (unit, row) summed over t in a fixed order; no atomics.  So a row's result depends only on its own inputs and the
 * set of units: call the unit chunks in increasing order, each over any split of the rows, and the bits do not
 * change.  finish_units > 0 (the total U of the walk, on the call with its last units): d_attr [rows, 2, F] =
 * (importance = acc / (U T), shift = acc / U) and d_mu_mean [rows] = acc / U, divided in double and rounded to fp32
 * once.  d_mu_units [n_units, rows] (may be NULL): each unit's mu.  The g block is transient workspace scratch (16.4 kB
 * per (unit, row)): size the chunks with bnn_posterior_saliency_workspace_bytes(cfg, n_units, rows) (0 for bad
 * arguments), which is non-decreasing in both counts: a workspace sized for (n_units, rows) serves every call of at most
 * n_units units and rows rows (a walk's smaller remainder chunks included); it begins with this call's summary draws [n_units, rows, 2L], which bnn_predict reproduces bit for bit
 * when given them as d_eps.  BNN_E_ARG: null pointer, n_units outside [1, 65535], rows outside [1, 2^30), unit or row indices past
 * 2^32, finish_units neither 0 nor in [n_units, 2^32); BNN_E_CONFIG: T != 100 or F != 41; BNN_E_ALIGN: d_workspace not
 * 16-byte, d_acc not 8-byte or a float array not 4-byte aligned; every check runs before the device is touched. */
size_t bnn_posterior_saliency_workspace_bytes(const bnn_model_config* cfg, int32_t n_units, int64_t rows);
int bnn_posterior_saliency(const bnn_model_config* cfg, int32_t n_units, const float* d_theta, int64_t unit0,
                           const float* d_x, int64_t rows, int64_t row0, uint64_t seed, double* d_acc, int32_t first,
                           int64_t finish_units, float* d_attr, float* d_mu_mean, float* d_mu_units, void* d_workspace,
                           void* stream);

/* The Philox draws bnn_train_step makes for (seed, step) when its eps pointers are NULL. */
int bnn_train_noise(const bnn_model_config* cfg, int32_t n_seeds, int64_t B, uint64_t seed, uint64_t step,
                    float* d_eps_in, float* d_eps12, float* d_eps_sum, void* stream);

/* lossfnc(x, y, noisy_val=False) (:579-583) without gradients, for n_units weight vectors at once:
 * validation_step (:787-799) evaluates it at the current weights and at w_avg.
 * d_loss_sum [n_units]: sum over the B systems of _lossfnc.  d_eps [n_units,B,2L] or NULL (Philox).
 * d_out_mu_sd [n_units,B,2] receives the predictions; when NULL, d_workspace must hold
 * n_units*B*2 floats. */
int bnn_eval_loss(const bnn_model_config* cfg, const float* d_x, const float* d_y, int64_t B,
                  const float* d_theta_packed, int64_t n_units, const float* d_eps, uint64_t seed,
                  float* d_out_mu_sd, float* d_loss_sum, void* d_workspace, void* stream);

/* ---------------------------------------------------------------------------------------
 * SWAGModel.aggregate_model (:763-785) for n_seeds models at once.
 *   w_avg  <- (w_avg*n + w)/(n+1),  w2_avg <- (w2_avg*n + w*w)/(n+1)   (first call: w, w*w)
 *   when the model has no deviation column yet, or current_epoch % c == 0 (:776-782):
 *   append w as the newest column of pre_D[s] ([d,K] row-major, columns oldest -> newest,
 *   d_n_cols[s] valid columns; the oldest is dropped beyond K).
 * d_w [n_seeds,d] current flat weights; d_n_models / d_n_cols [n_seeds] int32, updated in place.
 */
int bnn_swag_collect(const float* d_w, int64_t d, int32_t n_seeds, int32_t K, float* d_w_avg,
                     float* d_w2_avg, float* d_pre_D, int32_t* d_n_models, int32_t* d_n_cols,
                     int32_t current_epoch, int32_t c, void* stream);

/* bnn_swag_collect that leaves halted seeds untouched: a seed with d_halted_at[s] >= 0 (the word of
 * bnn_train_step_seeds_halt) keeps its w_avg, w2_avg, pre_D, n_models and n_cols; the other seeds collect as with
 * bnn_swag_collect, which is this entry with no halt word.  A seed that halts during an epoch is therefore not collected
 * at the end of it, like a reference run that ended mid-epoch.  BNN_E_ARG: a null pointer or bad size; BNN_E_ALIGN:
 * d_halted_at not 8-byte aligned; both before the device is touched. */
int bnn_swag_collect_halt(const float* d_w, int64_t d, int32_t n_seeds, int32_t K, float* d_w_avg,
                          float* d_w2_avg, float* d_pre_D, int32_t* d_n_models, int32_t* d_n_cols,
                          int32_t current_epoch, int32_t c, const int64_t* d_halted_at, void* stream);

/* ---------------------------------------------------------------------------------------
 * Input packing, the step upstream of bnn_predict: data_setup_kernel (figures/spock/regression.py:183-213)
 * + ssX.transform (:144) + .float() (:145).  d_tseries [N,T,26] float64 raw time series (already sub-sampled
 * to T steps, :141), d_masses [N,3] float64 planet/star mass ratios (:142), d_ss_mean / d_ss_scale [41]
 * float64 StandardScaler constants (spock_reg_model.py:934-955) -> d_x [N,T,41] float32: 3 non-finite flags,
 * nan_to_num, (cos, sin) of the 9 angle columns, standardisation; float64 arithmetic like numpy.
 */
int bnn_pack_inputs(const double* d_tseries, const double* d_masses, const double* d_ss_mean,
                    const double* d_ss_scale, int64_t n_systems, int32_t n_times, float* d_x, void* stream);

/* ---------------------------------------------------------------------------------------
 * Posterior post-processing, the step downstream of bnn_predict (figures/main_figures.py:167-277,
 * figures/multiswag_5_planet.py:306-481), on the system-major prediction block d_pred [n_rows, U, 2]
 * (row = system * n_trios + trio; U weight samples):
 * bnn_sample_instability: fast_truncnorm(mu, std, left, nsamp) -- the first of nsamp normal draws
 *   x = z*std + mu that exceeds `left` (the first draw if none does) -- and, where the result is >= 9, a fresh
 *   draw from the analytic prior on [9, 100] by inverse CDF.  Philox keyed on (seed; row_offset + row, unit).
 *   d_t [n_rows, U].
 * bnn_summarize_instability: per system, over the U weight samples of min-over-trios(t): d_stats [N, 8] =
 *   average, median, percentiles 84, 16, 97.5, 2.5 (numpy 'linear'), then the median over weight samples of
 *   mu* = min over trios of mu and of the std of that trio ("median of dists", main_figures.py:276-277).
 *   U <= 32768: shared-memory bitonic sort; larger U (30 models x 2000 samples): exact 3-pass radix select.
 */
int bnn_sample_instability(const float* d_pred, int64_t n_rows, int64_t n_units, uint64_t seed, int64_t row_offset,
                           float left, int32_t nsamp, float* d_t, void* stream);
int bnn_summarize_instability(const float* d_t, const float* d_pred, int64_t n_systems, int32_t n_trios,
                              int32_t n_units, float* d_stats, void* stream);

/* Held-out score of the ensemble on the same system-major block d_pred [n_systems, U, 2] (one trio per system) against
 * the labels d_y [n_systems, 2] (the two labels of a system, as bnn_nll_fwd_bwd takes them).  loss[n,u] is
 * bnn_nll_fwd_bwd's per-system loss of (mu, sd) = d_pred[n,u] and d_y[n] (VarModel._lossfnc, non-finite terms -> 100).
 * d_score [n_systems, 2]:
 *   [0] lpd      = log((1/U) sum_u exp(-loss[n,u])), the log predictive density of the label pair in nats;
 *   [1] mean_nll = (1/U) sum_u loss[n,u].
 * Both are evaluated in double (lpd as m + log sum_u exp(-loss - m) - log U, m = max_u -loss) and rounded to fp32 once.
 * A row's result depends on that row's inputs only, through a fixed reduction order: any row slice of a block scores
 * bit-identically, and repeated calls are bit-identical.  Pointers need only 8-byte alignment, so a slice at any row is
 * accepted.  BNN_E_ARG: null pointer, n_systems <= 0 or >= 2^31, n_units <= 0 or >= 2^32; checked before the device. */
int bnn_score_labels(const float* d_pred, int64_t n_systems, int64_t n_units, const float* d_y, float* d_score,
                     void* stream);

/* Survival probability per system from the sampled times d_t [n_systems * n_trios, U] that bnn_sample_instability
 * writes (row = system * n_trios + trio).  tmin[n,u] is the min over trios exactly as bnn_summarize_instability takes
 * it: fminf from +inf, so a unit whose trio draws are all NaN counts as +inf.  For the J = n_thresholds host values
 * h_thresholds (log10 orbits, any order, duplicates and +-inf allowed):
 *   d_surv [n_systems, J]:  surv[n,j] = #{u : tmin[n,u] > h_thresholds[j]} / U   (strict comparison),
 * the count exact, converted once as (float)((double)count / U).  It is a Monte Carlo estimate of P(T_inst > thr) with
 * standard error sqrt(S (1 - S) / U), from the same draws as the summary's percentiles.  The thresholds travel in the
 * kernel's parameters (no device copy).  A row's result depends on that row only, and repeated calls are bit-identical.
 * d_t and d_surv need only 4-byte alignment, so a row slice at any offset is accepted.  BNN_E_ARG: null pointer,
 * n_systems <= 0 or >= 2^31, n_units <= 0 or >= 2^32, n_trios < 1, n_thresholds outside [1, 64], a NaN threshold;
 * checked before the device. */
int bnn_survival_instability(const float* d_t, int64_t n_systems, int32_t n_trios, int64_t n_units,
                             const float* h_thresholds, int32_t n_thresholds, float* d_surv, void* stream);

/* Catalogues of mixed planet counts: the same summary and survival for systems with different numbers of trio rows.
 * d_row_offsets is a DEVICE int64 array [n_systems + 1]; system n owns the rows d_row_offsets[n] - d_row_offsets[0] ..
 * d_row_offsets[n+1] - d_row_offsets[0] - 1 of d_t (and of d_pred), so its trio count is
 * c[n] = d_row_offsets[n+1] - d_row_offsets[n], and the min over trios runs over those c[n] rows.  Rows are counted from
 * d_row_offsets[0]: a slice of systems [a, b) of a catalogue passes a view of the catalogue's offsets (&off[a]) with its
 * own d_t / d_pred rows, with no rebased copy.  With every c[n] = R the results equal bnn_summarize_instability /
 * bnn_survival_instability with n_trios = R bit for bit, and a system's result depends on its own rows only.
 * The offsets are NOT validated on the device (that would need a synchronisation): a system whose count is <= 0 gets a
 * NaN row (all 8 statistics, all J survival columns), so such an offsets array has a defined result; offsets that are
 * non-decreasing but run past the rows given read outside the block, and are the caller's to prevent (the Python layer
 * validates the counts before it uploads them).  Variant choice (sort up to U = 32768, radix select beyond,
 * bnn_set_summary_variant) is as for bnn_summarize_instability.  BNN_E_ARG as for the uniform entries plus a null
 * d_row_offsets; BNN_E_ALIGN: d_row_offsets not 8-byte aligned (and, for survival, d_t / d_surv not 4-byte aligned);
 * every check runs before the device is touched. */
int bnn_summarize_instability_ragged(const float* d_t, const float* d_pred, int64_t n_systems, const int64_t* d_row_offsets,
                                     int32_t n_units, float* d_stats, void* stream);
int bnn_survival_instability_ragged(const float* d_t, int64_t n_systems, const int64_t* d_row_offsets, int64_t n_units,
                                    const float* h_thresholds, int32_t n_thresholds, float* d_surv, void* stream);

/* Which trio sets each system's instability time, from the sampled times d_t [rows, U] that bnn_sample_instability
 * writes.  tmin[n,u] is the min over system n's trio rows exactly as bnn_summarize_instability takes it (fminf from
 * +inf).  The winner at unit u is the FIRST of the system's rows r with t[r,u] == tmin[n,u] (ties go to the earlier
 * trio; +inf is an ordinary value, so when every non-NaN draw is +inf the first +inf row wins); a unit whose draws are
 * all NaN has no winner.  For each trio row r of system n:
 *   d_first [rows]:  first[r] = #{u : r wins unit u} / U,
 * the count exact, converted once as (float)((double)count / U); so sum_r first[r] = (U - #all-NaN units) / U.  Rows
 * are system-major: system * n_trios + trio for the uniform entry, the offsets' rows for the ragged one (counted from
 * d_row_offsets[0] as in bnn_survival_instability_ragged, so a slice of systems passes a view of the catalogue's
 * offsets and its own d_t / d_first rows).  A system's result depends on its own rows only, and repeated calls are
 * bit-identical.  At most 1024 trio rows per system: a ragged system with a larger count gets NaN rows, one with a count
 * <= 0 owns no rows and nothing is written.  d_t and d_first need only 4-byte alignment.  BNN_E_ARG: null pointer,
 * n_systems <= 0 or >= 2^31, n_units <= 0 or >= 2^32, n_trios < 1 or > 1024; BNN_E_ALIGN: d_t / d_first not 4-byte or
 * d_row_offsets not 8-byte aligned; every check runs before the device is touched. */
int bnn_first_trio_instability(const float* d_t, int64_t n_systems, int32_t n_trios, int64_t n_units, float* d_first,
                               void* stream);
int bnn_first_trio_instability_ragged(const float* d_t, int64_t n_systems, const int64_t* d_row_offsets, int64_t n_units,
                                      float* d_first, void* stream);

/* Variance decomposition of every row of the system-major block d_pred [n_rows, U, 2] (row = system * n_trios + trio).
 * Unit u = k * S + s is weight sample s of model k, S = units_per_model, M = U / S models; mu_{k,s} and sigma_{k,s} are
 * its predicted normal in log10 orbits.  With m_k = (1/S) sum_s mu_{k,s} and mean = (1/M) sum_k m_k, d_out [n_rows, 5]:
 *   [0] mean_mu        = mean
 *   [1] aleatoric      = (1/U) sum_u sigma_u^2
 *   [2] epistemic      = between_models + within_models (added in double) = (1/U) sum_u (mu_u - mean)^2
 *   [3] between_models = (1/M) sum_k (m_k - mean)^2
 *   [4] within_models  = (1/M) sum_k (1/S) sum_s (mu_{k,s} - m_k)^2
 * Population (ddof = 0) moments: by the law of total variance the equal-weight mixture of the U normals has variance
 * aleatoric + epistemic.  They describe the untruncated per-unit normals, not the sampled times of
 * bnn_sample_instability (truncated at 4, resampled above 9, min over trios).  Two-pass in double (model means first,
 * then deviations), rounded to fp32 once: between_models is exactly 0 when M = 1, within_models when S = 1, and both
 * and epistemic when all mu of a row are equal.  A non-finite mu in a row makes columns 0, 2, 3, 4 NaN; a non-finite
 * sigma makes column 1 NaN.  A row's result depends on that row only (fixed reduction order, no atomics): any row slice
 * reproduces its rows bit for bit, and repeated calls are bit-identical.  BNN_E_ARG: null pointer, n_rows <= 0 or
 * >= 2^31, n_units <= 0 or >= 2^32, units_per_model < 1, n_units not a multiple of units_per_model, more than 1024
 * models; BNN_E_ALIGN: d_pred not 8-byte or d_out not 4-byte aligned; checked before the device. */
int bnn_decompose_uncertainty(const float* d_pred, int64_t n_rows, int64_t n_units, int64_t units_per_model,
                              float* d_out, void* stream);

/* K8: the short N-body integration from initial orbits to the model's raw inputs (csrc/nbody.cu; DESIGN.md section
 * K8).  d_elements [n_systems, n_planets, 7] holds per planet, from the inside out, (m / M_star, a, e, inc, Omega,
 * varpi, lambda): Jacobi elements (primary = star + interior planets, mu = G (M_interior + m)), G = M_star = 1.  Each
 * system is integrated on its own by WHFast-style Wisdom-Holman (drift-kick-drift, Jacobi interaction kick, Gauss f
 * and g drift, no corrector) with dt = dt_frac min_i P_i (1 - e_i)^(3/2) / sqrt(1 + e_i), and sampled at the first
 * step boundary t >= t_k = 10 k n_orbits / 999 P1, k = 0..99 (P1: the innermost initial period).  Per adjacent trio
 * (i, i+1, i+2), rows system-major and trio-minor (the tseries / masses layout bnn_pack_inputs takes):
 *   d_tseries [n_systems (n_planets - 2), 100, 26]: t / P1, 0 x 7, then per trio planet (a / a_{i,0}, e, inc, Omega,
 *     varpi, theta), angles in [0, 2 pi), a_{i,0} the initial a of the trio's innermost planet;
 *   d_masses [n_systems (n_planets - 2), 3]: (m_i, m_{i+1}, m_{i+2});
 *   d_log10_t_unstable [n_systems]: log10(t / P1) at the first step whose kick sees two planets nearer than the sum
 *     of their Hill radii a_{j,0} (m_j / 3)^(1/3), or after which a Jacobi orbit is unbound; NaN when the system
 *     reaches its last output.  An unstable system's rows from that step on are NaN.
 * Element values are not checked on the device: a system with a planet of a <= 0, e outside [0, 1), m < 0 or a
 * non-finite value, or whose own step count exceeds 2^31, gets NaN rows and NaN log10_t_unstable (its masses are
 * still copied).  A system's bits depend on its own elements only.  BNN_E_ARG: null pointer, n_systems outside
 * [1, 2^31), n_planets outside [3, 8], n_orbits or dt_frac not finite and > 0, (990 / 999) n_orbits / dt_frac > 2^31
 * (every system's step count is at least that); BNN_E_ALIGN: an array not 8-byte aligned; every check runs before the
 * device is touched. */
int bnn_integrate_orbits(const double* d_elements, int64_t n_systems, int32_t n_planets, double n_orbits, double dt_frac,
                         double* d_tseries, double* d_masses, double* d_log10_t_unstable, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* BNNCHAOS_H_ */

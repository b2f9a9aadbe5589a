// K5: SWAG moment collection for several seed models at once.
//
// Reference: SWAGModel.aggregate_model (/root/reference/spock_reg_model.py:763-785):
//   first call:  w_avg = w, w2_avg = w^2, pre_D = w[:,None]
//   later:       w_avg = (w_avg*n + w)/(n+1), w2_avg likewise;
//                if current_epoch % c == 0: append w as newest column, keep the last K
//   n += 1
// pre_D is kept as a fixed [d,K] row-major buffer with n_cols valid columns (oldest first),
// so a full buffer is exactly the tensor save_swag writes (:917).  HBM-bound, tiny.
#include "common.cuh"

namespace bnn {

// halted_at (may be null): a seed with halted_at[s] >= 0 (bnn_train_step_seeds_halt) is left untouched, here and in
// swag_bump_kernel.
__global__ void swag_collect_kernel(const float* __restrict__ w, int64_t d, int K, float* __restrict__ w_avg,
                                    float* __restrict__ w2_avg, float* __restrict__ pre_D,
                                    const int32_t* __restrict__ n_models, const int32_t* __restrict__ n_cols,
                                    int current_epoch, int c, const int64_t* __restrict__ halted_at) {
    const int s = blockIdx.y;
    const int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (j >= d || (halted_at && halted_at[s] >= 0)) return;
    const int n = n_models[s];
    const int nc = n_cols[s];
    const int64_t o = (int64_t)s * d + j;
    const float cw = w[o];
    const float cw2 = __fmul_rn(cw, cw);
    if (n == 0) {
        w_avg[o] = cw;
        w2_avg[o] = cw2;
    } else {
        const float nf = (float)n, n1 = (float)(n + 1);
        w_avg[o] = __fdiv_rn(__fadd_rn(__fmul_rn(w_avg[o], nf), cw), n1);
        w2_avg[o] = __fdiv_rn(__fadd_rn(__fmul_rn(w2_avg[o], nf), cw2), n1);
    }
    const bool record = (nc == 0) || (current_epoch % c == 0);
    if (record) {
        float* row = pre_D + o * K;
        if (nc < K) {
            row[nc] = cw;
        } else {
            for (int k = 0; k + 1 < K; ++k) row[k] = row[k + 1];
            row[K - 1] = cw;
        }
    }
}

__global__ void swag_bump_kernel(int32_t* n_models, int32_t* n_cols, int n_seeds, int K, int current_epoch, int c,
                                 const int64_t* __restrict__ halted_at) {
    const int s = threadIdx.x + blockIdx.x * blockDim.x;
    if (s >= n_seeds || (halted_at && halted_at[s] >= 0)) return;
    const int nc = n_cols[s];
    if ((nc == 0) || (current_epoch % c == 0)) n_cols[s] = min(nc + 1, K);
    n_models[s] += 1;
}

// bnn_swag_collect (halted_at null) and bnn_swag_collect_halt; every argument check runs before the device is touched
static int swag_collect(const char* who, const float* d_w, int64_t d, int32_t n_seeds, int32_t K, float* d_w_avg,
                        float* d_w2_avg, float* d_pre_D, int32_t* d_n_models, int32_t* d_n_cols, int32_t current_epoch,
                        int32_t c, bool halt, const int64_t* d_halted_at, cudaStream_t st) {
    BNN_REQUIRE(d_w && d_w_avg && d_w2_avg && d_pre_D && d_n_models && d_n_cols && (!halt || d_halted_at), BNN_E_ARG,
                "%s: null pointer", who);
    BNN_REQUIRE(d > 0 && n_seeds > 0 && n_seeds < 65536 && K >= 1 && c >= 1, BNN_E_ARG,
                "%s: bad sizes (d=%lld seeds=%d K=%d c=%d)", who, (long long)d, n_seeds, K, c);
    BNN_REQUIRE(((uintptr_t)d_halted_at & 7u) == 0, BNN_E_ALIGN, "%s: d_halted_at must be 8-byte aligned", who);
    int rc = check_device();
    if (rc != BNN_OK) return rc;
    const int threads = 256;
    dim3 grid((unsigned)((d + threads - 1) / threads), (unsigned)n_seeds);
    swag_collect_kernel<<<grid, threads, 0, st>>>(d_w, d, K, d_w_avg, d_w2_avg, d_pre_D, d_n_models, d_n_cols,
                                                  current_epoch, c, d_halted_at);
    BNN_CUDA(cudaGetLastError());
    swag_bump_kernel<<<(n_seeds + 127) / 128, 128, 0, st>>>(d_n_models, d_n_cols, n_seeds, K, current_epoch, c, d_halted_at);
    BNN_CUDA(cudaGetLastError());
    return BNN_OK;
}

}  // namespace bnn

extern "C" int bnn_swag_collect(const float* d_w, int64_t d, int32_t n_seeds, int32_t K, float* d_w_avg,
                                float* d_w2_avg, float* d_pre_D, int32_t* d_n_models, int32_t* d_n_cols,
                                int32_t current_epoch, int32_t c, void* stream) {
    return bnn::swag_collect("bnn_swag_collect", d_w, d, n_seeds, K, d_w_avg, d_w2_avg, d_pre_D, d_n_models, d_n_cols,
                             current_epoch, c, false, nullptr, (cudaStream_t)stream);
}

extern "C" int bnn_swag_collect_halt(const float* d_w, int64_t d, int32_t n_seeds, int32_t K, float* d_w_avg,
                                     float* d_w2_avg, float* d_pre_D, int32_t* d_n_models, int32_t* d_n_cols,
                                     int32_t current_epoch, int32_t c, const int64_t* d_halted_at, void* stream) {
    return bnn::swag_collect("bnn_swag_collect_halt", d_w, d, n_seeds, K, d_w_avg, d_w2_avg, d_pre_D, d_n_models,
                             d_n_cols, current_epoch, c, true, d_halted_at, (cudaStream_t)stream);
}

// ---------------------------------------------------------------------------------------
// K6: input packing -- the step immediately upstream of the predictive kernel (SURVEY 8f rank 2).
//
// Reference: data_setup_kernel (/root/reference/figures/spock/regression.py:183-213) followed by
// ssX.transform (:144, float64 sklearn StandardScaler) and torch.tensor(X).float() (:145):
//   raw row = [26 time-series columns | 3 masses | isnotfinite(col 3), (col 6), (col 7)]   (32 columns)
//   nan_to_num(posinf=0, neginf=0);  angle columns {11,12,13,17,18,19,23,24,25} -> (cos, sin)    (41 columns)
//   x = float32((X - mean) / scale)        (all arithmetic in float64, like numpy)
// HBM-bound: 232 B read + 164 B written per time-step row.
// ---------------------------------------------------------------------------------------
namespace bnn {

constexpr int PACK_ROWS = 32;  // time-step rows per CTA tile

// out column of raw column j: every angle column before j adds one
__device__ __forceinline__ int pack_out_col(int j) {
    int oc = j;
    if (j > 11) oc += min(j - 11, 3);
    if (j > 17) oc += min(j - 17, 3);
    if (j > 23) oc += min(j - 23, 3);
    return oc;
}

// One CTA = 32 consecutive rows: coalesced load of the 32 x 26 doubles into shared memory, then warp-homogeneous
// work lists (288 sincos items first, 736 plain items after) so that the fp64 trigonometry does not diverge against
// the copy columns, results staged in shared memory and written back as one contiguous 32 x 41 float block.
__global__ void __launch_bounds__(256) pack_inputs_kernel(const double* __restrict__ ts, const double* __restrict__ mass,
                                                          const double* __restrict__ mean, const double* __restrict__ scale,
                                                          int64_t n_rows, int T, float* __restrict__ x) {
    __shared__ double raw[PACK_ROWS][26];
    __shared__ float o[PACK_ROWS][41];
    __shared__ double sm_mean[41], sm_scale[41];
    const int64_t row0 = (int64_t)blockIdx.x * PACK_ROWS;
    const int nr = (int)min((int64_t)PACK_ROWS, n_rows - row0);
    for (int i = threadIdx.x; i < nr * 26; i += 256) (&raw[0][0])[i] = ts[row0 * 26 + i];
    if (threadIdx.x < 41) { sm_mean[threadIdx.x] = mean[threadIdx.x]; sm_scale[threadIdx.x] = scale[threadIdx.x]; }
    __syncthreads();
    // angle columns {11,12,13,17,18,19,23,24,25}: (cos, sin)
    for (int w = threadIdx.x; w < nr * 9; w += 256) {
        const int r = w / 9, a = w - r * 9;
        const int j = 11 + (a / 3) * 6 + a % 3;
        double v = raw[r][j];
        if (!isfinite(v)) v = 0.0;  // np.nan_to_num(posinf=0.0, neginf=0.0): NaN -> 0 too
        double sn, cs;
        sincos(v, &sn, &cs);
        const int oc = pack_out_col(j);
        o[r][oc] = (float)((cs - sm_mean[oc]) / sm_scale[oc]);
        o[r][oc + 1] = (float)((sn - sm_mean[oc + 1]) / sm_scale[oc + 1]);
    }
    // the 23 plain columns: 17 time-series columns, 3 masses, 3 non-finite flags
    for (int w = threadIdx.x; w < nr * 23; w += 256) {
        const int r = w / 23, p = w - r * 23;
        // p -> raw column: 0..10, 14..16, 20..22, 26..31
        const int j = p < 11 ? p : (p < 14 ? p + 3 : (p < 17 ? p + 6 : p + 9));
        double v;
        if (j < 26) {
            v = raw[r][j];
        } else if (j < 29) {
            v = mass[((row0 + r) / T) * 3 + (j - 26)];
        } else {
            const int src = (j == 29) ? 3 : (j == 30 ? 6 : 7);
            v = isfinite(raw[r][src]) ? 0.0 : 1.0;  // flags are taken before nan_to_num
        }
        if (!isfinite(v)) v = 0.0;
        const int oc = pack_out_col(j);
        o[r][oc] = (float)((v - sm_mean[oc]) / sm_scale[oc]);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < nr * 41; i += 256) x[row0 * 41 + i] = (&o[0][0])[i];
}

}  // namespace bnn

extern "C" int bnn_pack_inputs(const double* d_tseries, const double* d_masses, const double* d_ss_mean,
                               const double* d_ss_scale, int64_t n_systems, int32_t n_times, float* d_x, void* stream) {
    using namespace bnn;
    int rc = check_device();
    if (rc != BNN_OK) return rc;
    BNN_REQUIRE(d_tseries && d_masses && d_ss_mean && d_ss_scale && d_x, BNN_E_ARG, "bnn_pack_inputs: null pointer");
    BNN_REQUIRE(n_systems > 0 && n_times > 0, BNN_E_ARG, "bnn_pack_inputs: empty input");
    const int64_t blocks = (n_systems * n_times + PACK_ROWS - 1) / PACK_ROWS;
    BNN_REQUIRE(blocks < (1ll << 31), BNN_E_ARG, "bnn_pack_inputs: too many rows for one launch");
    pack_inputs_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(d_tseries, d_masses, d_ss_mean, d_ss_scale,
                                                                          n_systems * n_times, n_times, d_x);
    BNN_CUDA(cudaGetLastError());
    return BNN_OK;
}

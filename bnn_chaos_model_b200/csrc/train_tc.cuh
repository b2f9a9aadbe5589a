// K4-TC: the fused SWAG training step with ALL EIGHT GEMMs of a system on the 5th-generation tensor cores
// (tcgen05.mma kind::tf32, accumulators in tensor memory).  Included by train.cu, namespace bnn::train.
//
// Same math, boundary and partial-gradient format as train_fwd_bwd3_kernel (derivation in the header of train.cu;
// reference: /root/reference/spock_reg_model.py:486-528 forward(noisy_val=True), :547-593 loss + KL, :722-732
// training_step).  Why a new kernel: the CUDA-core formulations stall at a third of the FP32 roofline (v3 is
// latency-bound at 3 warps per scheduler, v4 shared-memory-bound; DESIGN.md section 4) because every FMA operand
// crosses the 32-words-per-cycle shared-memory -> register path.  tcgen05 reads its operands from shared / tensor
// memory itself; the CUDA cores only run the per-row epilogues.
//
// One CTA per SM owns one seed (its weights are staged ONCE as tf32 hi / lo B operands, natural and transposed) and
// walks that seed's systems.  A system is one M = 128 tile (100 time-step rows = TMEM lanes 0..99).  Two systems are
// in flight ("slots"); per slot four row warps (thread = row = TMEM lane):
//   stage   x'' (image of the noisy input, see producers) -> exact x' -> hi / lo -> tcgen05.st A
//   L1, L2  tcgen05.ld D -> + bias -> ReLU -> hi / lo -> tcgen05.st A of the next layer, and the tf32-rounded
//           activation into shared memory [row quad][feature][4 rows] -- the K-major layout, K = rows, that the
//           weight-gradient GEMMs contract over
//   L3      D + bias -> f (registers + shared memory) -> two-pass pooling, sampled summary statistics, regress_nn
//           forward, truncated-normal NLL, regress_nn backward (the 128 threads of the slot, six short phases; head
//           weight gradients are deferred through one record per system exactly as in v3)
//   g_f     -> hi / lo -> A, rounded -> shared memory;   issue  dW2 += g_f^T [h2 | 1]   and   g_a2 = g_f W2
//   g_a2    D . [h2 > 0] -> A, shared memory (over h2);  issue  dW1 += g_a2^T [h1 | 1]  and   g_a1 = g_a2 W1
//   g_a1    D . [h1 > 0] -> shared memory (over h1);     issue  [dW0 | E | db0] += g_a1^T [x' | n | 1]
// The g_x = g_a1 W0 GEMM of the CUDA-core kernels is gone: dlv_in[c] = 1/2 sum_r g_x[r][c] n[r][c] (n = x' - mask(x))
// = 1/2 sum_j W0[j][c] E[j][c] with E = g_a1^T n, which rides in the same MMAs as dW0 (n is stored only for the live
// columns: for a zeroed column mask(x) = 0, so n = x' and E = dW0).  The bias gradients are the "ones" column.
//
// Numerics.  Row GEMMs (forward and the two activation-gradient GEMMs): 3xTF32 (a = a_hi + a_lo, w = w_hi + w_lo;
// a_lo w_hi + a_hi w_lo + a_hi w_hi, corrections first -- the accumulator rounds toward zero), as in the predictive
// kernel: loss and logged scalars match the fp32 reference to 1e-5.  Weight-gradient GEMMs: ONE tf32 pass on operands
// rounded to NEAREST (stored as bits + 0x1000: the tensor core drops the 13 low mantissa bits, so the bias turns its
// truncation into round-to-nearest-ties-away, and bits - 0x1000 gives the exact fp32 value back to the row threads).
// The rounding errors are unbiased and independent per (row, feature); over the B x T rows of a batch they average
// out: measured against the reference's autograd, max |dg| / max |g| = 2e-5 at B = 64 (three golden steps) and 2e-6 at
// B = 2000, against the 2e-4 tolerance of tests/test_gpu_train.py (the hardware's own truncation would be biased:
// 8e-5).  tools/dw_precision.py reproduces the study on the CPU.
//
// Warp roles (16 warps, 512 threads, one CTA per SM):
//   0..7   row warps: slot = w / 4, TMEM lane quadrant = w % 4
//   8      issuer: the only thread that issues tcgen05.mma (one in-order stream: the three weight-gradient
//          accumulators are shared by both slots and are updated in strict tile order, so a step is bit-reproducible)
//          and the bulk copies (cp.async.bulk) of the input images
//   9..15  producers: draw the Philox input noise up to four tiles ahead and write the tile's IMAGE -- exactly the
//          bytes of the slot's shared-memory input area: [row quad][x''(41) | n''(live) | 1][4 rows], eps1 | eps2,
//          summary noise, labels -- into an L2-resident ring; one 30 kB bulk copy brings it in when the slot is free.
// Tensor memory (512 columns): slot s: A_hi [144 s, +48) A_lo [+48, +96) D [+96, +144); acc0 [288, 288 + N0) =
// [dW0 | E | db0], acc1 [384, 432) = [dW1 | db1], acc2 [432, 480) = [dW2 | db2]; lanes = output feature j.
#pragma once
#include "tc.cuh"

namespace bnn {
namespace train {
namespace tcx {

constexpr int T = 100, F = 41;
constexpr int NQ = 26, RQ = 25;          // row quads: 104 rows = 13 k-steps of 8 rows; 25 hold data
constexpr int KS_ROWS = 13;
constexpr int PHH = 41;                  // features per quad of the h1 / h2 arrays: 40 + the ones column
constexpr int PGF = 21;                  // features per quad of the f / g_f array (20 + 1 pad: odd pitch, conflict-free)
constexpr int SMALLF = 96;               // tail of an image: eps1|eps2 [40], summary noise [40], labels [2], pad
constexpr int IM_E12 = 0, IM_ESN = 40, IM_Y = 80;
constexpr int NST = 8;                   // depth of the L2 image ring
constexpr int NSLOT = 2;
constexpr int XG = 11;                   // 4-column groups of x (44 columns, 41 real)
constexpr int W_ISSUE = 8, W_PROD = 10, NPW = 6, NWARP = 16, NTHR_TC = NWARP * 32;   // 512 threads: 128 registers each
constexpr int TM_AHI = 0, TM_ALO = 48, TM_D = 96, TM_SLOT = 144, TM_ACC0 = 288, TM_ACC1 = 384, TM_ACC2 = 432;
constexpr int SVF = 512;                 // head scratch per slot (layout: the V3_* enum of train_v3.cuh)
// B-operand shapes (canonical K-major chunks [k/4][n][4]; only the real n rows are stored, the MMA's surplus rows
// read the next chunk and land in D columns nobody loads)
constexpr int K1C = 12, K2C = 10, KB2C = 6;   // 16-byte K chunks: layer 1 (48), layers 2 / 3 and g_a1 (40), g_a2 (24)

enum Phase { PH_X = 0, PH_L1, PH_L2, PH_L3, PH_B2, PH_B1, PH_DW0, PH_END };

struct Bars {
    uint64_t a_ready[NSLOT];   // 128 row threads: operands of the slot's next phase are in place
    uint64_t a_ready0[NSLOT];  // the same for layer 1 of the slot's NEXT tile: its stage does not wait for the issuer to have
                               // consumed the previous tile's last a_ready phase, and an mbarrier can only be one phase ahead
    uint64_t d_ready[NSLOT];   // tcgen05.commit of the slot's phase
    uint64_t x_free[NSLOT];    // tcgen05.commit of the slot's last phase: its shared-memory areas may be overwritten
    uint64_t x_full[NSLOT];    // bulk copy of the slot's image landed (the issuer waits for it before the last phase)
    uint64_t img_full[NST];    // producers finished the image of ring stage i
    uint64_t img_free[NST];    // ring stage i has been read by the slot's 128 row threads AND copied out by the bulk copy
    uint32_t tmem_base;
    int turn[3];               // tile whose weight-gradient MMAs may be issued next into acc0 / acc1 / acc2 (two issuers)
};

struct SmemTC {
    int NL, PX, N0, img_floats, stage_floats;
    int xa[NSLOT], h1[NSLOT], h2[NSLOT], gf[NSLOT], sv[NSLOT];
    int B1h, B1l, B2h, B2l, B3h, B3l, W2Th, W2Tl, W1Th, W1Tl, bias, V0, V1, V2, cb, consts, lidx, bars, total;
    __host__ __device__ SmemTC(uint64_t zero_mask) {
        NL = 0;
        for (int c = 0; c < F; ++c) NL += ((zero_mask >> c) & 1ull) ? 0 : 1;
        PX = (F + NL + 1) | 1;                       // x'' | n''(live) | ones (| pad): odd pitch, conflict-free
        N0 = (F + NL + 1 + 15) & ~15;
        img_floats = NQ * PX * 4 + SMALLF;            // what the bulk copy brings into the slot's input area
        stage_floats = img_floats + XG * 4 * NQ * 4;  // + x'' once more as [4-column group][row][4]: the row threads' own
                                                      //   stage reads (11 fully coalesced 16-byte loads per thread)
        int o = 0;
        for (int s = 0; s < NSLOT; ++s) {
            xa[s] = o; o += img_floats;
            h1[s] = o; o += NQ * PHH * 4;
            h2[s] = o; o += NQ * PHH * 4;
            gf[s] = o; o += NQ * PGF * 4;
            sv[s] = o; o += SVF;
        }
        B1h = o; o += K1C * H * 4;  B1l = o; o += K1C * H * 4;
        B2h = o; o += K2C * H * 4;  B2l = o; o += K2C * H * 4;
        B3h = o; o += K2C * L * 4;  B3l = o; o += K2C * L * 4;
        W2Th = o; o += KB2C * H * 4; W2Tl = o; o += KB2C * H * 4;
        W1Th = o; o += K2C * H * 4;  W1Tl = o; o += K2C * H * 4;
        bias = o; o += 128;          // b0[40] pad 8 | b1[40] pad 8 | b2[20] pad 12
        V0 = o; o += H * S2;
        V1 = o; o += H * H;
        V2 = o; o += 2 * H;
        cb = o; o += 2 * H + 4;
        consts = o; o += C3_TOTAL;
        lidx = o; o += 64;           // int: image column of n for feature c, or -1
        o = (o + 3) & ~3;
        bars = o; o += (int)((sizeof(Bars) + 3) / 4);
        // the M = 128 A descriptors of the weight-gradient GEMMs read 2 kB per row quad: 1.4 kB past the end of the
        // array for the last quads; everything up to here is followed by valid shared memory, the tail pad covers h1[1]
        total = o + 512;
    }
    __host__ __device__ bool fits() const { return (size_t)total * 4 <= 227 * 1024 && N0 <= 96; }
};

__device__ __forceinline__ uint32_t rn_bias(float v) { return __float_as_uint(v) + 0x1000u; }

// v -> (tf32 hi, fp32 lo) for the 3xTF32 A operand, and the biased word for shared memory
__device__ __forceinline__ void split3(float v, uint32_t& hi, uint32_t& lo, uint32_t& biased) {
    biased = rn_bias(v);
    hi = biased & 0xFFFFE000u;
    lo = __float_as_uint(v - __uint_as_float(hi));
}

// ---- MMA issue (one elected lane of the converged issuer warp) ----
template <int N, int KS>
__device__ __forceinline__ void issue_ts3(uint32_t d, uint32_t ahi, uint32_t alo, uint32_t bh_addr, uint32_t bl_addr,
                                          uint32_t chunk_bytes) {
    constexpr uint32_t idesc = idesc_tf32(128, N);
    const uint64_t dh = smem_desc_kmajor(bh_addr, chunk_bytes, 128u), dl = smem_desc_kmajor(bl_addr, chunk_bytes, 128u);
    const uint64_t step = (uint64_t)(2u * chunk_bytes) >> 4;
    if (elect_one_sync()) {
#pragma unroll
        for (int ks = 0; ks < KS; ++ks) mma_tf32_ts(d, alo + 8 * ks, dh + ks * step, idesc, ks > 0);
#pragma unroll
        for (int ks = 0; ks < KS; ++ks) mma_tf32_ts(d, ahi + 8 * ks, dl + ks * step, idesc, true);
#pragma unroll
        for (int ks = 0; ks < KS; ++ks) mma_tf32_ts(d, ahi + 8 * ks, dh + ks * step, idesc, true);
    }
    __syncwarp();
}
// D = A_hi (W_lo + W_hi): the activation-gradient GEMMs, A rounded to nearest (one operand word), W split
template <int N, int KS>
__device__ __forceinline__ void issue_ts2(uint32_t d, uint32_t ahi, uint32_t bh_addr, uint32_t bl_addr, uint32_t chunk_bytes) {
    constexpr uint32_t idesc = idesc_tf32(128, N);
    const uint64_t dh = smem_desc_kmajor(bh_addr, chunk_bytes, 128u), dl = smem_desc_kmajor(bl_addr, chunk_bytes, 128u);
    const uint64_t step = (uint64_t)(2u * chunk_bytes) >> 4;
    if (elect_one_sync()) {
#pragma unroll
        for (int ks = 0; ks < KS; ++ks) mma_tf32_ts(d, ahi + 8 * ks, dl + ks * step, idesc, ks > 0);
#pragma unroll
        for (int ks = 0; ks < KS; ++ks) mma_tf32_ts(d, ahi + 8 * ks, dh + ks * step, idesc, true);
    }
    __syncwarp();
}
// acc (+)= A^T B over the 104 rows: A [row quad][feature][4] with pa features per quad, B likewise with pb
__device__ __forceinline__ void issue_ss_rows(uint32_t acc, uint32_t a_addr, uint32_t pa, uint32_t b_addr, uint32_t pb,
                                              uint32_t idesc, bool first) {
    const uint64_t ad = smem_desc_kmajor(a_addr, pa * 16u, 128u), bd = smem_desc_kmajor(b_addr, pb * 16u, 128u);
    const uint64_t sa = (uint64_t)(2u * pa), sb = (uint64_t)(2u * pb);   // two quads per k-step, in 16-byte units
    if (elect_one_sync()) {
#pragma unroll
        for (int ks = 0; ks < KS_ROWS; ++ks) mma_tf32_ss(acc, ad + ks * sa, bd + ks * sb, idesc, !(first && ks == 0));
    }
    __syncwarp();
}

// ---- producers: the image of one tile ----
struct ProdTC {
    const float* X; const float* eps_in; const float* Y; const float* eps12; const float* eps_sum;
    const float* nsc; const int* lidx;
    uint64_t key, zero_mask; int64_t sb; int row, b, step, PX, NL, rm_off;   // rm_off: float offset of the [group][row][4] copy
};

// items (row quad q < 25, feature c): 4 normals (Philox block q * F + c, box_muller_fast) for rows 4q..4q+3 of column c
template <int NR>
__device__ __forceinline__ void produce_items(const ProdTC& a, float* __restrict__ img, int first, int stride) {
    float xv[NR][4], ev[NR][4];
    uint4 ctr[NR];
    int qs[NR], cs[NR];
    bool ok[NR];
#pragma unroll
    for (int k = 0; k < NR; ++k) {
        const int id0 = first + stride * k;
        ok[k] = id0 < RQ * F;
        const int id = ok[k] ? id0 : RQ * F - 1;
        const int q = id / F, c = id - q * F;
        qs[k] = q; cs[k] = c;
        ctr[k] = make_uint4((uint32_t)id, (uint32_t)a.b, (uint32_t)a.step, STREAM_EPS_IN);
        const float* xs = a.X + ((int64_t)a.row * T + 4 * q) * F + c;
#pragma unroll
        for (int u = 0; u < 4; ++u) xv[k][u] = __ldg(xs + u * F);
    }
    if (a.eps_in) {
#pragma unroll
        for (int k = 0; k < NR; ++k) {
            const float* es = a.eps_in + (a.sb * T + 4 * qs[k]) * (int64_t)F + cs[k];
#pragma unroll
            for (int u = 0; u < 4; ++u) ev[k][u] = __ldg(es + u * F);
        }
    } else {
        constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
        uint32_t k0 = (uint32_t)a.key, k1 = (uint32_t)(a.key >> 32);
#pragma unroll
        for (int r = 0; r < 10; ++r) {
#pragma unroll
            for (int k = 0; k < NR; ++k) {
                const uint4 c = ctr[k];
                const uint32_t hi0 = __umulhi(M0, c.x), lo0 = M0 * c.x;
                const uint32_t hi1 = __umulhi(M1, c.z), lo1 = M1 * c.z;
                ctr[k] = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
            }
            k0 += W0;
            k1 += W1;
        }
#pragma unroll
        for (int k = 0; k < NR; ++k) {
            const float4 n4 = box_muller_fast(ctr[k]);
            ev[k][0] = n4.x; ev[k][1] = n4.y; ev[k][2] = n4.z; ev[k][3] = n4.w;
        }
    }
#pragma unroll
    for (int k = 0; k < NR; ++k) {
        if (!ok[k]) continue;
        const int c = cs[k];
        const bool zeroed = (a.zero_mask >> c) & 1ull;
        const float sc = a.nsc[c];
        uint32_t xb[4], nb[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            float x = xv[k][u];
            if (zeroed) x = __fsub_rn(x, x);                       // x - mask keeps NaN (:452-478)
            const float xp = __fadd_rn(x, __fmul_rn(ev[k][u], sc));   // :444-446
            xb[u] = rn_bias(xp);
            nb[u] = rn_bias(__fsub_rn(xp, x));
        }
        float* dst = img + (qs[k] * a.PX + c) * 4;
        *reinterpret_cast<uint4*>(dst) = make_uint4(xb[0], xb[1], xb[2], xb[3]);
        uint32_t* rm = reinterpret_cast<uint32_t*>(img) + a.rm_off + (((c >> 2) * (4 * NQ) + 4 * qs[k]) * 4 + (c & 3));
#pragma unroll
        for (int u = 0; u < 4; ++u) rm[4 * u] = xb[u];
        const int li = a.lidx[c];
        if (li >= 0) *reinterpret_cast<uint4*>(img + (qs[k] * a.PX + li) * 4) = make_uint4(nb[0], nb[1], nb[2], nb[3]);
    }
}

__device__ __forceinline__ void produce_rest(const ProdTC& a, float* __restrict__ img, int p, int NPRODT) {
    // ones column (and the pad column when PX is padded) of the 25 data quads, the whole pad quad, the small inputs
    const int c1 = F + a.NL;
    for (int i = p; i < RQ * (a.PX - c1); i += NPRODT) {
        const int q = i / (a.PX - c1), c = c1 + i - q * (a.PX - c1);
        const float v = c == c1 ? 1.0f : 0.f;
        *reinterpret_cast<float4*>(img + (q * a.PX + c) * 4) = make_float4(v, v, v, v);
    }
    for (int i = p; i < a.PX; i += NPRODT) *reinterpret_cast<float4*>(img + (RQ * a.PX + i) * 4) = make_float4(0.f, 0.f, 0.f, 0.f);
    float* sm_out = img + NQ * a.PX * 4;
    if (p < 10) {
        float4 e, c;
        if (a.eps12) {
            e = __ldg(reinterpret_cast<const float4*>(a.eps12 + a.sb * S2) + p);
            c = __ldg(reinterpret_cast<const float4*>(a.eps_sum + a.sb * S2) + p);
        } else {
            e = philox_normal4(a.key, STREAM_EPS, (uint32_t)a.b, (uint32_t)a.step, (uint32_t)p);
            c = philox_normal4(a.key, STREAM_EPS_SUM, (uint32_t)a.b, (uint32_t)a.step, (uint32_t)p);
        }
        reinterpret_cast<float4*>(sm_out + IM_E12)[p] = e;
        reinterpret_cast<float4*>(sm_out + IM_ESN)[p] = c;
    } else if (p == 10) {
        float2 y = __ldg(reinterpret_cast<const float2*>(a.Y) + a.row);
        *reinterpret_cast<float4*>(sm_out + IM_Y) = make_float4(y.x, y.y, 0.f, 0.f);
    } else if (p >= 11 && p < 14) {
        *reinterpret_cast<float4*>(sm_out + IM_Y + 4 * (p - 10)) = make_float4(0.f, 0.f, 0.f, 0.f);
    }
}

// ---- row-thread epilogues, NC consecutive columns of this thread's row -------------------------------------------
// hidden layer: v = relu(d + bias) -> A (tf32 hi, fp32 lo) and the biased word (bits + 0x1000) into arow[col * 4]
template <int NC>
__device__ __forceinline__ void hidden_cols(const uint32_t (&d)[NC], const float* __restrict__ bl, float* __restrict__ arow,
                                            bool stored, uint32_t t_hi, uint32_t t_lo) {
    uint32_t hi[NC], lo[NC];
#pragma unroll
    for (int g4 = 0; g4 < NC / 4; ++g4) {
        const ulonglong2 b = *reinterpret_cast<const ulonglong2*>(bl + 4 * g4);
        const u64 v01 = add2(pack2(__uint_as_float(d[4 * g4]), __uint_as_float(d[4 * g4 + 1])), b.x);
        const u64 v23 = add2(pack2(__uint_as_float(d[4 * g4 + 2]), __uint_as_float(d[4 * g4 + 3])), b.y);
        float v[4];
        unpack2(v01, v[0], v[1]);
        unpack2(v23, v[2], v[3]);
        uint32_t hb[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            v[u] = relu_nan(v[u]);
            const uint32_t bz = rn_bias(v[u]);
            hb[u] = bz & 0xFFFFE000u;
            hi[4 * g4 + u] = hb[u];
            if (stored) arow[(4 * g4 + u) * 4] = __uint_as_float(bz);
        }
        const u64 l01 = sub2(pack2(v[0], v[1]), pack2(__uint_as_float(hb[0]), __uint_as_float(hb[1])));
        const u64 l23 = sub2(pack2(v[2], v[3]), pack2(__uint_as_float(hb[2]), __uint_as_float(hb[3])));
        float l[4];
        unpack2(l01, l[0], l[1]);
        unpack2(l23, l[2], l[3]);
#pragma unroll
        for (int u = 0; u < 4; ++u) lo[4 * g4 + u] = __float_as_uint(l[u]);
    }
    if constexpr (NC == 16) {
        tmem_st16(t_hi, hi);
        tmem_st16(t_lo, lo);
    } else {
        tmem_st8(t_hi, hi);
        tmem_st8(t_lo, lo);
    }
}
// activation gradient: g = d . [h > 0] (h's biased word sits in arow[col * 4]; +0 is 0x1000) -> the biased word of g over
// it, and (TM) the rounded g as the A operand of the next activation-gradient GEMM (single word: 2-term product)
template <int NC, bool TM>
__device__ __forceinline__ void grad_cols(const uint32_t (&d)[NC], float* __restrict__ arow, bool stored, uint32_t t_hi) {
    uint32_t hi[NC];
    uint32_t hw[NC];
#pragma unroll
    for (int j = 0; j < NC; ++j) hw[j] = stored ? __float_as_uint(arow[j * 4]) : 0u;
#pragma unroll
    for (int j = 0; j < NC; ++j) {
        const uint32_t g = hw[j] > 0x1000u ? d[j] : 0u;
        const uint32_t bz = g + 0x1000u;
        hi[j] = bz & 0xFFFFE000u;
        if (stored) arow[j * 4] = __uint_as_float(bz);
    }
    if constexpr (TM) {
        if constexpr (NC == 16) tmem_st16(t_hi, hi);
        else tmem_st8(t_hi, hi);
    }
}

__device__ __forceinline__ void slot_sync(int slot) { named_sync(3 + slot, 128); }

// per-role cycle stamps of CTA (0, 0) (make train_timeline; read back with bnn_train_timeline): row thread 0 -> slots
// 0..12 (x wait | stage | D wait, epilogue x 2 | D wait | head: last phase | g_f | D wait | g_a2 | D wait | g_a1) and 13..18
// (head: f store | pooling | V0 | V1 | output + NLL | V1^T), issuer of slot 0 -> 20 (loop) 21 (inside issue), producer
// warp 0 -> 22 (work) 23 (waiting for a free ring stage)
#ifdef BNN_TRAIN_TIMELINE
#define TCT_DECL long long tct_prev = tl_clock(); unsigned long long tct[19] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0}
#define TCT(i) do { if (tid == 0) { const long long t_ = tl_clock(); tct[i] += (unsigned long long)(t_ - tct_prev); tct_prev = t_; } } while (0)
#define TCT_FLUSH do { if (tid == 0 && blockIdx.x == 0 && blockIdx.y == 0) for (int i_ = 0; i_ < 19; ++i_) g_train_tl[i_] = tct[i_]; } while (0)
#else
#define TCT_DECL do { } while (0)
#define TCT(i) do { } while (0)
#define TCT_FLUSH do { } while (0)
#endif

}  // namespace tcx

__global__ void __launch_bounds__(tcx::NTHR_TC, 1) train_tc_kernel(const Params prm) {
    using namespace tcx;
    extern __shared__ __align__(16) float sm[];
    const SmemTC L_(prm.zero_mask);
    const FlatLayout fl(F);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int sidx = prm.seed0 + (int)blockIdx.y;
    const float* th = prm.theta + (int64_t)sidx * fl.d;
    Bars* bars = reinterpret_cast<Bars*>(sm + L_.bars);
    float* cst = sm + L_.consts;
    float* V0s = sm + L_.V0; float* V1s = sm + L_.V1; float* V2s = sm + L_.V2; float* cbs = sm + L_.cb;
    int* lidx = reinterpret_cast<int*>(sm + L_.lidx);
    const int PX = L_.PX, NL = L_.NL;
    const int n_k = (prm.B - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;   // this CTA's systems (tiles)

    // ---- one-time setup: weights as tf32 hi / lo B operands, head weights, constants, barriers, TMEM ----
    for (int i = tid; i < L_.total; i += NTHR_TC)
        if (i < L_.B1h || i >= L_.bars + (int)((sizeof(Bars) + 3) / 4)) sm[i] = 0.f;   // activation areas, tail pad
    auto put = [&](int oh, int ol, int idx, float w) {
        const float hi = __uint_as_float((__float_as_uint(w) + 0x1000u) & 0xFFFFE000u);
        sm[oh + idx] = hi;
        sm[ol + idx] = tf32_rna(w - hi);
    };
    for (int i = tid; i < K1C * 4 * H; i += NTHR_TC) {          // layer 1: B[n][k] = W0[n][k], k < 48
        const int k = i / H, n = i - k * H;
        put(L_.B1h, L_.B1l, ((k >> 2) * H + n) * 4 + (k & 3), k < F ? __ldg(th + fl.W0 + n * F + k) : 0.f);
    }
    for (int i = tid; i < H * H; i += NTHR_TC) {
        const int k = i / H, n = i - k * H;
        put(L_.B2h, L_.B2l, ((k >> 2) * H + n) * 4 + (k & 3), __ldg(th + fl.W1 + n * H + k));     // layer 2: W1[n][k]
        put(L_.W1Th, L_.W1Tl, ((k >> 2) * H + n) * 4 + (k & 3), __ldg(th + fl.W1 + k * H + n));   // g_a1: B[n][j] = W1[j][n]
        V1s[i] = __ldg(th + fl.V1 + i);
        V0s[i] = __ldg(th + fl.V0 + i);   // H * S2 == H * H
    }
    for (int i = tid; i < H * L; i += NTHR_TC) {                // layer 3: B[n][k] = W2[n][k], n < 20
        const int k = i / L, n = i - k * L;
        put(L_.B3h, L_.B3l, ((k >> 2) * L + n) * 4 + (k & 3), __ldg(th + fl.W2 + n * H + k));
    }
    for (int i = tid; i < KB2C * 4 * H; i += NTHR_TC) {         // g_a2: B[n][c] = W2[c][n], c < 24
        const int c = i / H, n = i - c * H;
        put(L_.W2Th, L_.W2Tl, ((c >> 2) * H + n) * 4 + (c & 3), c < L ? __ldg(th + fl.W2 + c * H + n) : 0.f);
    }
    if (tid < H) {
        sm[L_.bias + tid] = __ldg(th + fl.b0 + tid);
        sm[L_.bias + 48 + tid] = __ldg(th + fl.b1 + tid);
        cbs[tid] = __ldg(th + fl.c0 + tid); cbs[H + tid] = __ldg(th + fl.c1 + tid);
    }
    if (tid < L) sm[L_.bias + 96 + tid] = __ldg(th + fl.b2 + tid);
    if (tid < 2 * H) V2s[tid] = __ldg(th + fl.V2 + tid);
    if (tid < 2) cbs[2 * H + tid] = __ldg(th + fl.c2 + tid);
    if (tid < S2) {
        const float lv = __ldg(th + fl.lv_sum + tid);
        cst[C3_LVS + tid] = lv;
        cst[C3_ELVH + tid] = expf(__fdiv_rn(lv, 2.0f));
        cst[C3_KLC + tid] = expf(lv) - lv - 1.0f;
    }
    if (tid < F) cst[C3_NSC + tid] = expf(__fdiv_rn(__ldg(th + fl.lv_in + tid), 2.0f));
    if (tid < 64) {
        int li = -1;
        if (tid < F && !((prm.zero_mask >> tid) & 1ull)) {
            li = F;
            for (int c = 0; c < tid; ++c) li += ((prm.zero_mask >> c) & 1ull) ? 0 : 1;
        }
        lidx[tid] = li;
    }
    if (tid == 0) {
        for (int s = 0; s < NSLOT; ++s) {
            mbar_init(&bars->a_ready[s], 128);
            mbar_init(&bars->a_ready0[s], 128);
            mbar_init(&bars->d_ready[s], 1);
            mbar_init(&bars->x_free[s], 1);
            mbar_init(&bars->x_full[s], 1);
        }
        for (int s = 0; s < NST; ++s) { mbar_init(&bars->img_full[s], 96); mbar_init(&bars->img_free[s], 128 + 1); }
        bars->turn[0] = bars->turn[1] = bars->turn[2] = 0;
        mbar_init_fence();
    }
    if (warp == 0) { tmem_alloc(&bars->tmem_base, 512); tmem_relinquish(); }
    __syncthreads();
    // the ones column of the h1 / h2 arrays (column 40 of the 25 data quads; the pad quad stays zero)
    for (int i = tid; i < NSLOT * 2 * RQ; i += NTHR_TC) {
        const int s = i / (2 * RQ), r = i - s * 2 * RQ, a = r / RQ, q = r - a * RQ;
        float* base = sm + (a ? L_.h2[s] : L_.h1[s]);
        *reinterpret_cast<float4*>(base + (q * PHH + H) * 4) = make_float4(1.f, 1.f, 1.f, 1.f);
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = bars->tmem_base;
    const uint64_t key = seed_key(prm.seed, sidx);
    float* ring = prm.xprod + ((int64_t)sidx * prm.n_cta + blockIdx.x) * (int64_t)(NST * L_.stage_floats);
    const uint32_t img_bytes = (uint32_t)L_.img_floats * 4u;

    float a_nll = 0.f, a_skl = 0.f;   // row threads: metric partial sums (lane 0 of the slot's warp 0 / the 20 pooling leaders)

    if (warp >= W_PROD) {
        // =================================================================================================
        // Producers: warp w draws the images of tiles w, w + NPW, ... ALONE (the work is latency-bound -- Philox chains,
        // DRAM loads of the rows -- so six independent tile streams beat six warps sharing one tile), up to NST tiles ahead
        // =================================================================================================
        const int pw = warp - W_PROD;
#ifdef BNN_TRAIN_TIMELINE
        long long tp_wait = 0, tp_work = 0;
#endif
        // tiles 0 and 1 (the first tile of each slot) are drawn by three warps each, so that the pipeline starts after a
        // third of a warp's tile time; from tile 2 on every warp has its own stream: pw + 2, pw + 2 + NPW, ...
        for (int it = -1;; ++it) {
            const bool coop = it < 0;
            const int k = coop ? pw / 3 : NSLOT + pw + it * NPW;
            if (k >= n_k) { if (coop) continue; else break; }
            const int p0 = coop ? (pw % 3) * 32 + lane : lane, pstride = coop ? 96 : 32;
            const int st = k % NST;
#ifdef BNN_TRAIN_TIMELINE
            const long long tp0 = tl_clock();
#endif
            if (k >= NST) mbar_wait_backoff(&bars->img_free[st], (uint32_t)((k / NST - 1) & 1), 200);
#ifdef BNN_TRAIN_TIMELINE
            const long long tp1 = tl_clock();
#endif
            const int b = (int)blockIdx.x + k * (int)gridDim.x;
            ProdTC a;
            a.X = prm.X; a.eps_in = prm.eps_in; a.Y = prm.Y; a.eps12 = prm.eps12; a.eps_sum = prm.eps_sum;
            a.nsc = cst + C3_NSC; a.lidx = lidx; a.key = key; a.zero_mask = prm.zero_mask;
            a.sb = (int64_t)sidx * prm.B + b;
            a.row = prm.batch_index ? prm.batch_index[a.sb] : b;
            a.b = b; a.step = (int)prm.step; a.PX = PX; a.NL = NL; a.rm_off = L_.img_floats;
            float* img = ring + (int64_t)st * L_.stage_floats;
            {   // pull the rows of this warp's next tile into L2 (129 lines of 128 B per system)
                const int b2 = ((int)blockIdx.x) + (coop ? NSLOT + pw : k + NPW) * (int)gridDim.x;
                if (b2 < prm.B) {
                    const int64_t sb2 = (int64_t)sidx * prm.B + b2;
                    const int64_t r2 = prm.batch_index ? (int64_t)prm.batch_index[sb2] : (int64_t)b2;
                    for (int ln = lane; ln < 129; ln += 32) {
                        const char* p2 = reinterpret_cast<const char*>(prm.X + r2 * T * F) + 128 * ln;
                        asm volatile("prefetch.global.L2 [%0];" ::"l"(p2));
                    }
                }
            }
            produce_rest(a, img, p0, pstride);
#pragma unroll 1
            for (int i0 = 0; i0 < RQ * F; i0 += 4 * pstride) produce_items<4>(a, img, i0 + p0, pstride);   // 1025 items
            __threadfence();                            // the image is read back by the bulk-copy engine through L2
            mbar_arrive_n(&bars->img_full[st], coop ? 1u : 3u);   // 96 arrivals complete a stage: 3 warps, or one warp x 3
#ifdef BNN_TRAIN_TIMELINE
            tp_wait += tp1 - tp0; tp_work += tl_clock() - tp1;
#endif
        }
#ifdef BNN_TRAIN_TIMELINE
        if (pw == 0 && lane == 0 && blockIdx.x == 0 && blockIdx.y == 0) { g_train_tl[22] = tp_work; g_train_tl[23] = tp_wait; }
#endif
    } else if (warp >= W_ISSUE) {
        // =================================================================================================
        // Issuers: warp W_ISSUE + s issues every tcgen05.mma and the image bulk copy of slot s, in the slot's program order.
        // The three weight-gradient accumulators are shared by the slots: their MMAs take turns in strict tile order
        // (turn[] in shared memory, handed over with tcgen05 fences), so a step is bit-reproducible.
        // =================================================================================================
        const int s = warp - W_ISSUE;
        const uint32_t sbase = smem_u32(sm);
        const uint32_t idesc48 = idesc_tf32(128, 48), idesc0 = idesc_tf32(128, L_.N0);
        const uint32_t ts = tmem + (uint32_t)(s * TM_SLOT);
        const uint32_t d = ts + TM_D, ahi = ts + TM_AHI, alo = ts + TM_ALO;
        uint32_t pa = 0, pa0 = 0, pxf = 0, pxl = 0;
        volatile int* turn = bars->turn;
        auto take_turn = [&](int acc, int k) {
            while (turn[acc] != k) __nanosleep(20);
            __syncwarp();
            tc_fence_after();
        };
        auto pass_turn = [&](int acc, int k) {
            tc_fence_before();
            __syncwarp();
            if (lane == 0) { __threadfence_block(); turn[acc] = k + 1; }
        };
        auto commit = [&](uint64_t* bar) {
            if (elect_one_sync()) mma_commit(bar);
            __syncwarp();
        };
#ifdef BNN_TRAIN_TIMELINE
        const long long ti0 = tl_clock();
        long long ti_issue = 0;
#define TI_BEGIN const long long ti1_ = tl_clock()
#define TI_END ti_issue += tl_clock() - ti1_
#else
#define TI_BEGIN do { } while (0)
#define TI_END do { } while (0)
#endif
        for (int k = s; k < n_k; k += NSLOT) {
            const int st = k % NST;
            // the image of tile k -> the slot's input area (read only by the last phase): needs the weight-gradient MMAs of
            // the slot's previous tile (its last readers) complete and the image produced
            if (k >= NSLOT) { mbar_wait_backoff(&bars->x_free[s], pxf, 20); pxf ^= 1; }
            mbar_wait_backoff(&bars->img_full[st], (uint32_t)((k / NST) & 1), 20);
            if (lane == 0) {
                asm volatile("fence.proxy.async;" ::: "memory");   // producers' generic-proxy writes -> bulk-copy engine
                mbar_arrive_expect_tx(&bars->x_full[s], img_bytes);
                bulk_g2s(sm + L_.xa[s], ring + (int64_t)st * L_.stage_floats, img_bytes, &bars->x_full[s]);
            }
            __syncwarp();
            mbar_wait(&bars->a_ready0[s], pa0); pa0 ^= 1;
            tc_fence_after();
            { TI_BEGIN; issue_ts3<48, 6>(d, ahi, alo, sbase + 4u * L_.B1h, sbase + 4u * L_.B1l, H * 16u); commit(&bars->d_ready[s]); TI_END; }
            mbar_wait(&bars->a_ready[s], pa); pa ^= 1;
            tc_fence_after();
            { TI_BEGIN; issue_ts3<48, 5>(d, ahi, alo, sbase + 4u * L_.B2h, sbase + 4u * L_.B2l, H * 16u); commit(&bars->d_ready[s]); TI_END; }
            mbar_wait(&bars->a_ready[s], pa); pa ^= 1;
            tc_fence_after();
            { TI_BEGIN; issue_ts3<32, 5>(d, ahi, alo, sbase + 4u * L_.B3h, sbase + 4u * L_.B3l, L * 16u); commit(&bars->d_ready[s]); TI_END; }
            mbar_wait(&bars->a_ready[s], pa); pa ^= 1;
            tc_fence_after();
            issue_ts2<48, 3>(d, ahi, sbase + 4u * L_.W2Th, sbase + 4u * L_.W2Tl, H * 16u);   // g_a2 first: it gates the row threads
            take_turn(2, k);
            { TI_BEGIN; issue_ss_rows(tmem + TM_ACC2, sbase + 4u * L_.gf[s], PGF, sbase + 4u * L_.h2[s], PHH, idesc48, k == 0); TI_END; }
            commit(&bars->d_ready[s]);
            pass_turn(2, k);
            mbar_wait(&bars->a_ready[s], pa); pa ^= 1;
            tc_fence_after();
            issue_ts2<48, 5>(d, ahi, sbase + 4u * L_.W1Th, sbase + 4u * L_.W1Tl, H * 16u);
            take_turn(1, k);
            { TI_BEGIN; issue_ss_rows(tmem + TM_ACC1, sbase + 4u * L_.h2[s], PHH, sbase + 4u * L_.h1[s], PHH, idesc48, k == 0); TI_END; }
            commit(&bars->d_ready[s]);
            pass_turn(1, k);
            mbar_wait(&bars->a_ready[s], pa); pa ^= 1;
            mbar_wait_backoff(&bars->x_full[s], pxl, 20); pxl ^= 1;      // [x' | n | 1] has landed
            if (lane == 0) mbar_arrive(&bars->img_free[st]);              // ... so the ring stage is free (with the 128 row threads)
            tc_fence_after();
            take_turn(0, k);
            { TI_BEGIN; issue_ss_rows(tmem + TM_ACC0, sbase + 4u * L_.h1[s], PHH, sbase + 4u * L_.xa[s], (uint32_t)PX, idesc0, k == 0); TI_END; }
            commit(&bars->x_free[s]);
            pass_turn(0, k);
        }
#ifdef BNN_TRAIN_TIMELINE
        if (s == 0 && lane == 0 && blockIdx.x == 0 && blockIdx.y == 0) { g_train_tl[20] = tl_clock() - ti0; g_train_tl[21] = ti_issue; }
#endif
        // every MMA of the slot has completed once its last commit has arrived
        {
            const int n_s = (n_k - s + NSLOT - 1) / NSLOT;   // tiles of slot s
            if (n_s > 0) mbar_wait_backoff(&bars->x_free[s], (uint32_t)((n_s - 1) & 1), 100);
        }
    } else {
        // =================================================================================================
        // Row warps
        // =================================================================================================
        const int slot = warp >> 2, quad = warp & 3;
        const int r = quad * 32 + lane;                     // tile row of this thread = TMEM lane
        const int lt = tid - slot * 128;                    // thread index inside the slot
        const bool live = r < T, stored = r < 4 * NQ;
        const uint32_t tl = tmem + (uint32_t)(slot * TM_SLOT) + ((uint32_t)(quad * 32) << 16);
        float* xa = sm + L_.xa[slot];
        float* h1a = sm + L_.h1[slot];
        float* h2a = sm + L_.h2[slot];
        float* gfa = sm + L_.gf[slot];
        float* sv = sm + L_.sv[slot];
        const int rq = (r >> 2), rr = r & 3;
        const float* bias = sm + L_.bias;
        const float Tf = (float)T, Tm1 = (float)(T - 1);
        uint32_t pd = 0;

        auto wait_d = [&]() {
            if (quad == 0) {   // try_wait suspends the warp in hardware until the phase completes: no polling granularity
                mbar_wait(&bars->d_ready[slot], pd);
                pd ^= 1;
            }
            named_sync(1 + slot, 128);
            tc_fence_after();
        };
        // operands of the next phase are written: TMEM stores complete, shared-memory stores visible to the tensor core
        auto publish = [&](bool layer1 = false) {
            tc_wait_st();
            tc_fence_before();
            fence_proxy_async_smem();
            mbar_arrive(layer1 ? &bars->a_ready0[slot] : &bars->a_ready[slot]);
        };
        auto hidden_epilogue = [&](const float* bl, float* act) {
            uint32_t d0[16], d1[16], d2[8];
            tmem_ld16(tl + TM_D, d0);
            tmem_ld16(tl + TM_D + 16, d1);
            tmem_ld8(tl + TM_D + 32, d2);
            tc_wait_ld();
            float* arow = act + rq * PHH * 4 + rr;
            hidden_cols<16>(d0, bl, arow, stored, tl + TM_AHI, tl + TM_ALO);
            hidden_cols<16>(d1, bl + 16, arow + 64, stored, tl + TM_AHI + 16, tl + TM_ALO + 16);
            hidden_cols<8>(d2, bl + 32, arow + 128, stored, tl + TM_AHI + 32, tl + TM_ALO + 32);
        };
        auto grad_epilogue_tm = [&](float* act) {
            uint32_t d0[16], d1[16], d2[8];
            tmem_ld16(tl + TM_D, d0);
            tmem_ld16(tl + TM_D + 16, d1);
            tmem_ld8(tl + TM_D + 32, d2);
            tc_wait_ld();
            float* arow = act + rq * PHH * 4 + rr;
            grad_cols<16, true>(d0, arow, stored, tl + TM_AHI);
            grad_cols<16, true>(d1, arow + 64, stored, tl + TM_AHI + 16);
            grad_cols<8, true>(d2, arow + 128, stored, tl + TM_AHI + 32);
        };
        auto grad_epilogue_sm = [&](float* act) {   // chunk by chunk: the prefetched x'' words (41 registers) are live across it
            float* arow = act + rq * PHH * 4 + rr;
            {
                uint32_t d0[16];
                tmem_ld16(tl + TM_D, d0);
                tc_wait_ld();
                grad_cols<16, false>(d0, arow, stored, 0u);
            }
            {
                uint32_t d1[16];
                tmem_ld16(tl + TM_D + 16, d1);
                tc_wait_ld();
                grad_cols<16, false>(d1, arow + 64, stored, 0u);
            }
            {
                uint32_t d2[8];
                tmem_ld8(tl + TM_D + 32, d2);
                tc_wait_ld();
                grad_cols<8, false>(d2, arow + 128, stored, 0u);
            }
        };

        TCT_DECL;
        for (int k = slot; k < n_k; k += NSLOT) {
            const int b = (int)blockIdx.x + k * (int)gridDim.x;
            const int64_t sb = (int64_t)sidx * prm.B + b;
            // ---- P0: the producers have finished the image -> this row's x'' straight from the L2 ring (11 coalesced 16-byte
            // ld.global.cg: the stage is rewritten every NST tiles, L1 must not serve it) -> exact x' -> A of layer 1 (48
            // columns, 41 real; rows >= T and the K padding are zeros); the tile's small inputs -> head scratch ----
            const int st = k % NST;
            const float* img = ring + (int64_t)st * L_.stage_floats;
            if (lane == 0) mbar_wait_backoff(&bars->img_full[st], (uint32_t)((k / NST) & 1), 40);
            __syncwarp();
            TCT(0);
            {
                uint4 xg[XG];
                const uint4* xr = reinterpret_cast<const uint4*>(img + L_.img_floats) + min(r, 4 * NQ - 1);
#pragma unroll
                for (int g = 0; g < XG; ++g) xg[g] = __ldcg(xr + g * (4 * NQ));
                if (lt < 21)   // eps1 | eps2, summary noise, labels: 82 floats, contiguous in the image and in the scratch
                    *reinterpret_cast<float4*>(sv + V3_E12 + 4 * lt) = __ldcg(reinterpret_cast<const float4*>(img + NQ * PX * 4) + lt);
#pragma unroll
                for (int c0 = 0; c0 < 48; c0 += 16) {
                    uint32_t hi[16], lo[16];
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        const int c = c0 + j, g = c < 44 ? c >> 2 : 0;
                        const uint32_t w = (c & 3) == 0 ? xg[g].x : ((c & 3) == 1 ? xg[g].y : ((c & 3) == 2 ? xg[g].z : xg[g].w));
                        const uint32_t bz = (c < F && live) ? w : 0x1000u;
                        hi[j] = bz & 0xFFFFE000u;
                        lo[j] = __float_as_uint(__uint_as_float(bz - 0x1000u) - __uint_as_float(hi[j]));
                    }
                    tmem_st16(tl + TM_AHI + c0, hi);
                    tmem_st16(tl + TM_ALO + c0, lo);
                }
            }
            mbar_arrive(&bars->img_free[st]);   // this thread's part of the image is in registers / tensor memory
            publish(true);
            TCT(1);
            // ---- P1, P2: hidden layers ----
            wait_d();
            TCT(2);
            hidden_epilogue(bias, h1a);
            publish();
            TCT(3);
            wait_d();
            TCT(4);
            hidden_epilogue(bias + 48, h2a);
            publish();
            TCT(5);
            // ---- P3: latent rows f = D + b2 -> registers and shared memory (the pooling reads columns) ----
            wait_d();
            TCT(6);
            float f[L];
            {
                uint32_t d0[16], d1[8];
                tmem_ld16(tl + TM_D, d0);
                tmem_ld8(tl + TM_D + 16, d1);
                tc_wait_ld();
#pragma unroll
                for (int c = 0; c < L; ++c) {
                    const float dv = __uint_as_float(c < 16 ? d0[c < 16 ? c : 0] : d1[c >= 16 ? c - 16 : 0]);
                    f[c] = live ? dv + bias[96 + c] : 0.f;
                    if (stored) gfa[(rq * PGF + c) * 4 + rr] = f[c];
                }
            }
            slot_sync(slot);
            TCT(13);
            // ---- pooling per latent column: two-pass mean / unbiased variance (:418-419), sampled summary statistics ----
            if (quad < 3) {   // 80 pooling threads (column c, 4 parts); the branch is warp-uniform for the shuffles
                const int c = min(lt >> 2, L - 1), part = lt & 3;
                float4 v[7];
#pragma unroll
                for (int i = 0; i < 7; ++i)
                    v[i] = (part + 4 * i < RQ) ? *reinterpret_cast<const float4*>(gfa + ((part + 4 * i) * PGF + c) * 4)
                                               : make_float4(0.f, 0.f, 0.f, 0.f);
                float s = 0.f;
#pragma unroll
                for (int i = 0; i < 7; ++i) s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
                s += __shfl_xor_sync(0xffffffffu, s, 1);
                s += __shfl_xor_sync(0xffffffffu, s, 2);
                const float mean = __fdiv_rn(s, Tf);
                float m2 = 0.f;
#pragma unroll
                for (int i = 0; i < 7; ++i)
                    if (part + 4 * i < RQ) {
                        const float d0 = v[i].x - mean, d1 = v[i].y - mean, d2 = v[i].z - mean, d3 = v[i].w - mean;
                        m2 = fmaf(d0, d0, m2); m2 = fmaf(d1, d1, m2); m2 = fmaf(d2, d2, m2); m2 = fmaf(d3, d3, m2);
                    }
                m2 += __shfl_xor_sync(0xffffffffu, m2, 1);
                m2 += __shfl_xor_sync(0xffffffffu, m2, 2);
                if (part == 0 && lt < L * 4) {
                    const float sd = sqrtf(__fdiv_rn(m2, Tm1));
                    const float var = __fmul_rn(sd, sd);
                    const float sim = sqrtf(__fdiv_rn(var, Tf));                                   // :422
                    const float siv = sqrtf(__fdiv_rn(__fmul_rn(2.0f, __fmul_rn(var, var)), Tm1));   // :423
                    const float e1 = sv[V3_E12 + c], e2 = sv[V3_E12 + L + c];
                    const float mus = __fadd_rn(__fmul_rn(e1, sim), mean);                          // :426
                    const float vs = __fadd_rn(__fmul_rn(e2, siv), var);                            // :427
                    const float sds = sqrtf(__fadd_rn(fabsf(vs), 1e-5f));                           // :430
                    sv[V3_M + c] = mean; sv[V3_VAR + c] = var; sv[V3_SIM + c] = sim; sv[V3_SIV + c] = siv; sv[V3_VS + c] = vs;
                    sv[V3_S + c] = mus; sv[V3_S + L + c] = sds;
                    sv[V3_SP + c] = __fadd_rn(mus, __fmul_rn(sv[V3_ESN + c], cst[C3_ELVH + c]));
                    sv[V3_SP + L + c] = __fadd_rn(sds, __fmul_rn(sv[V3_ESN + L + c], cst[C3_ELVH + L + c]));
                    a_skl += 0.5f * (mus * mus + cst[C3_KLC + c]) + 0.5f * (sds * sds + cst[C3_KLC + L + c]);
                }
            }
            slot_sync(slot);
            TCT(14);
            // ---- regress_nn forward: 10 outputs per warp, three 14 / 13 / 13-term partial sums per output ----
            const int hj = quad * 10 + (lane % 10), hpart = min(lane / 10, 2);   // lanes 30, 31 shadow part 2 (results unused)
            {
                float a = 0.f;
#pragma unroll
                for (int i = 0; i < 14; ++i) {
                    const int kx = hpart + 3 * i;
                    if (kx < S2) a = fmaf(sv[V3_SP + kx], V0s[hj * S2 + kx], a);
                }
                const float a1 = __shfl_down_sync(0xffffffffu, a, 10), a2 = __shfl_down_sync(0xffffffffu, a, 20);
                if (lane < 10) sv[V3_R1 + hj] = relu_nan((a + a1) + a2 + cbs[hj]);
            }
            slot_sync(slot);
            TCT(15);
            {
                float a = 0.f;
#pragma unroll
                for (int i = 0; i < 14; ++i) {
                    const int kx = hpart + 3 * i;
                    if (kx < H) a = fmaf(sv[V3_R1 + kx], V1s[hj * H + kx], a);
                }
                const float a1 = __shfl_down_sync(0xffffffffu, a, 10), a2 = __shfl_down_sync(0xffffffffu, a, 20);
                if (lane < 10) sv[V3_R2 + hj] = relu_nan((a + a1) + a2 + cbs[H + hj]);
            }
            slot_sync(slot);
            TCT(16);
            // ---- output layer, soft clamp, truncated-normal NLL and its gradient (one warp), V2 backward ----
            float gr0 = 0.f, gr1 = 0.f;
            if (quad == 0) {
                const int o = lane >> 4, l16 = lane & 15;
                float a = 0.f;
                for (int kx = l16; kx < H; kx += 16) a = fmaf(sv[V3_R2 + kx], V2s[o * H + kx], a);
                a += __shfl_xor_sync(0xffffffffu, a, 1);
                a += __shfl_xor_sync(0xffffffffu, a, 2);
                a += __shfl_xor_sync(0xffffffffu, a, 4);
                a += __shfl_xor_sync(0xffffffffu, a, 8);
                const float r0 = __shfl_sync(0xffffffffu, a, 0) + cbs[2 * H];
                const float r1 = __shfl_sync(0xffffffffu, a, 16) + cbs[2 * H + 1];
                const float t0 = tanhf(r0), t1 = tanhf(r1);
                const float mu = __fadd_rn(__fmul_rn(__fmul_rn(0.5f, __fadd_rn(t0, 1.0f)), __fsub_rn(prm.hc.hi_mu, prm.hc.lo_mu)), prm.hc.lo_mu);
                const float sd = __fadd_rn(__fmul_rn(__fmul_rn(0.5f, __fadd_rn(t1, 1.0f)), __fsub_rn(prm.hc.hi_sd, prm.hc.lo_sd)), prm.hc.lo_sd);
                float l = 0.f, dm = 0.f, ds = 0.f;
                if (lane < 2) nll_terms(mu, sd, sv[V3_Y + lane], l, dm, ds);
                const float l1 = __shfl_sync(0xffffffffu, l, 1), dm1 = __shfl_sync(0xffffffffu, dm, 1), ds1 = __shfl_sync(0xffffffffu, ds, 1);
                if (lane == 0) {
                    a_nll += -(l + l1);
                    const float gmu = -(dm + dm1), gsd = -(ds + ds1);
                    gr0 = gmu * 0.5f * (prm.hc.hi_mu - prm.hc.lo_mu) * (1.0f - t0 * t0);
                    gr1 = gsd * 0.5f * (prm.hc.hi_sd - prm.hc.lo_sd) * (1.0f - t1 * t1);
                }
                gr0 = __shfl_sync(0xffffffffu, gr0, 0);
                gr1 = __shfl_sync(0xffffffffu, gr1, 0);
                for (int kx = lane; kx < H; kx += 32) {
                    const float g = gr0 * V2s[kx] + gr1 * V2s[H + kx];
                    sv[V3_G2 + kx] = sv[V3_R2 + kx] > 0.f ? g : 0.f;
                }
            }
            slot_sync(slot);
            TCT(17);
            {   // g_a1h[k] = (sum_j g_a2h[j] V1[j][k]) . [r1 > 0]
                float a = 0.f;
#pragma unroll
                for (int i = 0; i < 14; ++i) {
                    const int j = hpart + 3 * i;
                    if (j < H) a = fmaf(sv[V3_G2 + j], V1s[j * H + hj], a);
                }
                const float a1 = __shfl_down_sync(0xffffffffu, a, 10), a2 = __shfl_down_sync(0xffffffffu, a, 20);
                if (lane < 10) sv[V3_G1 + hj] = sv[V3_R1 + hj] > 0.f ? (a + a1) + a2 : 0.f;
            }
            slot_sync(slot);
            TCT(18);
            float* rec = prm.head_rec + sb * REC;
            {   // g_s'[k] = sum_j g_a1h[j] V0[j][k]; summary-noise log-variance gradient; KL gradient of s
                float a = 0.f;
#pragma unroll
                for (int i = 0; i < 14; ++i) {
                    const int j = hpart + 3 * i;
                    if (j < H) a = fmaf(sv[V3_G1 + j], V0s[j * S2 + hj], a);
                }
                const float a1 = __shfl_down_sync(0xffffffffu, a, 10), a2 = __shfl_down_sync(0xffffffffu, a, 20);
                if (lane < 10) {
                    const float g = (a + a1) + a2;
                    rec[R_DLVS + hj] = g * (0.5f * (sv[V3_ESN + hj] * cst[C3_ELVH + hj]));   // ds'/dlv = eps e^{lv/2} / 2
                    sv[V3_GS + hj] = g + prm.beta_out[blockIdx.y] * sv[V3_S + hj];
                }
                // the record of the deferred head outer products: s', r1, r2, g_a1h, g_a2h (complete since the last barrier)
                for (int i = lt; i < R_DLVS; i += 128) rec[i] = sv[V3_REC0 + i];
                if (lt == 0) { rec[R_GR] = gr0; rec[R_GR + 1] = gr1; }
            }
            slot_sync(slot);
            TCT(7);
            // ---- P5: g_f[t] = g_m / n + g_v 2 (f_t - m) / (n - 1); lanes 0..19 of every warp hold their column's coefficients ----
            {
                float cA = 0.f, cB = 0.f, cM = 0.f;
                if (lane < L) {
                    const int c = lane;
                    const float gmus = sv[V3_GS + c], gsds = sv[V3_GS + L + c];
                    const float vs = sv[V3_VS + c], sds = sv[V3_S + L + c], var = sv[V3_VAR + c];
                    const float sgn = vs > 0.f ? 1.0f : (vs < 0.f ? -1.0f : 0.f);
                    const float gvs = gsds * sgn / (2.0f * sds);
                    const float e1 = sv[V3_E12 + c], e2 = sv[V3_E12 + L + c];
                    const float gv = gmus * e1 / (2.0f * Tf * sv[V3_SIM + c]) +
                                     gvs * (1.0f + e2 * (2.0f * var) / (Tm1 * sv[V3_SIV + c]));
                    cA = gmus / Tf;
                    cB = 2.0f * gv / Tm1;
                    cM = sv[V3_M + c];
                }
                uint32_t hi0[16], hi1[8];
#pragma unroll
                for (int c = 0; c < L; ++c) {
                    const float A = __shfl_sync(0xffffffffu, cA, c), Bc = __shfl_sync(0xffffffffu, cB, c), m = __shfl_sync(0xffffffffu, cM, c);
                    const float g = live ? fmaf(Bc, f[c] - m, A) : 0.f;   // rows >= T: exact zeros (they ARE rows of the contraction)
                    const uint32_t bz = rn_bias(g), h_ = bz & 0xFFFFE000u;
                    if (c < 16) hi0[c < 16 ? c : 0] = h_;
                    else hi1[c >= 16 ? c - 16 : 0] = h_;
                    if (stored) gfa[(rq * PGF + c) * 4 + rr] = __uint_as_float(live ? bz : 0u);
                }
#pragma unroll
                for (int c = L - 16; c < 8; ++c) hi1[c] = 0u;
                tmem_st16(tl + TM_AHI, hi0);
                tmem_st8(tl + TM_AHI + 16, hi1);
            }
            publish();
            TCT(8);
            // ---- P6: g_a2 = (g_f W2) . [h2 > 0] -> A and over h2 ----
            wait_d();
            TCT(9);
            grad_epilogue_tm(h2a);
            publish();
            TCT(10);
            // ---- P7: g_a1 = (g_a2 W1) . [h1 > 0] -> over h1; the issuer then adds g_a1^T [x' | n | 1] ----
            wait_d();
            TCT(11);
            grad_epilogue_sm(h1a);
            publish();
            TCT(12);
        }
        TCT_FLUSH;
    }

    // =====================================================================================================
    // Epilogue: this CTA's partial gradient in flatten() order
    // =====================================================================================================
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    float* part = prm.partial + ((int64_t)sidx * prm.n_cta + blockIdx.x) * (fl.d + DPAD);
    float* red = sm;   // the activation areas are dead
    // (1) feature matrices, biases, E: lanes 0..39 of the accumulators (row warps 0 and 1 of slot 0 own those lanes)
    if (warp < 2) {   // tcgen05.ld is warp-collective: every lane loads, lanes j >= 40 store nothing
        const int j = warp * 32 + lane;
        const bool jv = j < H;
        const uint32_t ta = tmem + ((uint32_t)(warp * 32) << 16);
        const int N0 = L_.N0;
        for (int c0 = 0; c0 < N0; c0 += 8) {
            uint32_t v[8];
            tmem_ld8(ta + TM_ACC0 + c0, v);
            tc_wait_ld();
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int c = c0 + i;
                const float a = __uint_as_float(v[i]);
                if (!jv) continue;
                if (c < F) {
                    part[fl.W0 + j * F + c] = a;
                    if (lidx[c] < 0) red[j * 48 + c] = __ldg(th + fl.W0 + j * F + c) * a;   // zeroed column: n = x', E = dW0
                } else if (c < F + NL) {
                    int cc = 0;   // feature whose noise sits in image column c
                    for (int t = 0; t < F; ++t) if (lidx[t] == c) cc = t;
                    red[j * 48 + cc] = __ldg(th + fl.W0 + j * F + cc) * a;
                } else if (c == F + NL) {
                    part[fl.b0 + j] = a;
                }
            }
        }
        for (int c0 = 0; c0 < 48; c0 += 8) {
            uint32_t v[8];
            tmem_ld8(ta + TM_ACC1 + c0, v);
            tc_wait_ld();
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int c = c0 + i;
                if (!jv) continue;
                if (c < H) part[fl.W1 + j * H + c] = __uint_as_float(v[i]);
                else if (c == H) part[fl.b1 + j] = __uint_as_float(v[i]);
            }
        }
        if (warp == 0) {
            for (int c0 = 0; c0 < 48; c0 += 8) {
                uint32_t v[8];
                tmem_ld8(ta + TM_ACC2 + c0, v);
                tc_wait_ld();
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int c = c0 + i;
                    if (j >= L) continue;
                    if (c < H) part[fl.W2 + j * H + c] = __uint_as_float(v[i]);
                    else if (c == H) part[fl.b2 + j] = __uint_as_float(v[i]);
                }
            }
        }
    }
    // (3) metrics: per-thread partial sums of the row threads
    red[48 * 48 + tid] = (warp < 8) ? a_skl : 0.f;
    red[48 * 48 + NTHR_TC + tid] = (warp < 8) ? a_nll : 0.f;
    __syncthreads();
    if (tid < F) {   // dlv_in[c] = 1/2 sum_j W0[j][c] E[j][c], fixed order
        float s = 0.f;
        for (int j = 0; j < H; ++j) s += red[j * 48 + tid];
        part[fl.lv_in + tid] = 0.5f * s;
    }
    if (tid == 0) {
        float s = 0.f, n = 0.f;
        for (int i = 0; i < 8 * 32; ++i) { s += red[48 * 48 + i]; n += red[48 * 48 + NTHR_TC + i]; }
        part[fl.d + SLOT_NLL] = n;
        part[fl.d + SLOT_SKL] = s;
        for (int i = 2; i < DPAD; ++i) part[fl.d + i] = 0.f;
    }
    __syncthreads();
    // (4) head gradients from the records of this CTA's systems, in system order (same roles as v3, 416 threads)
    {
        constexpr int CH = 128;
        const int jbh = tid / 10, kb = tid % 10;
        float aV0[2][4] = {}, aV1[2][4] = {};
        float s0 = 0.f, s1 = 0.f;
        for (int c0i = 0; c0i < n_k; c0i += CH) {
            const int nc = min(CH, n_k - c0i);
            for (int i = tid; i < nc * (REC / 4); i += NTHR_TC) {
                const int s = c0i + i / (REC / 4), w = i % (REC / 4);
                const int bsys = (int)blockIdx.x + (int)gridDim.x * s;
                reinterpret_cast<float4*>(red)[i] =
                    __ldcg(reinterpret_cast<const float4*>(prm.head_rec + ((int64_t)sidx * prm.B + bsys) * REC) + w);
            }
            __syncthreads();
            if (tid < 200) {
                for (int s = 0; s < nc; ++s) {
                    const float* rcd = red + s * REC;
#pragma unroll
                    for (int jj = 0; jj < 2; ++jj)
#pragma unroll
                        for (int q4 = 0; q4 < 4; ++q4) {
                            aV0[jj][q4] = fmaf(rcd[R_G1 + 2 * jbh + jj], rcd[R_SP + kb + 10 * q4], aV0[jj][q4]);
                            aV1[jj][q4] = fmaf(rcd[R_G2 + 2 * jbh + jj], rcd[R_R1 + kb + 10 * q4], aV1[jj][q4]);
                        }
                }
            } else if (tid < 240) {
                for (int s = 0; s < nc; ++s) { s0 += red[s * REC + R_G1 + tid - 200]; s1 += red[s * REC + R_G2 + tid - 200]; }
            } else if (tid < 320) {
                const int o = (tid - 240) / H, kx = (tid - 240) % H;
                for (int s = 0; s < nc; ++s) s0 = fmaf(red[s * REC + R_GR + o], red[s * REC + R_R2 + kx], s0);
            } else if (tid < 322) {
                for (int s = 0; s < nc; ++s) s0 += red[s * REC + R_GR + tid - 320];
            } else if (tid < 322 + S2) {
                for (int s = 0; s < nc; ++s) s0 += red[s * REC + R_DLVS + tid - 322];
            }
            __syncthreads();
        }
        if (tid < 200) {
#pragma unroll
            for (int jj = 0; jj < 2; ++jj)
#pragma unroll
                for (int q4 = 0; q4 < 4; ++q4) {
                    part[fl.V0 + (2 * jbh + jj) * S2 + kb + 10 * q4] = aV0[jj][q4];
                    part[fl.V1 + (2 * jbh + jj) * H + kb + 10 * q4] = aV1[jj][q4];
                }
        } else if (tid < 240) {
            part[fl.c0 + tid - 200] = s0;
            part[fl.c1 + tid - 200] = s1;
        } else if (tid < 320) {
            part[fl.V2 + tid - 240] = s0;
        } else if (tid < 322) {
            part[fl.c2 + tid - 320] = s0;
        } else if (tid < 322 + S2) {
            part[fl.lv_sum + tid - 322] = s0;
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem, 512);
}

}  // namespace train
}  // namespace bnn

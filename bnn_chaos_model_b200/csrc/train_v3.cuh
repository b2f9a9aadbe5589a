// K4 v3: the fused training forward + backward with large register tiles (included by train.cu, namespace bnn::train).
//
// Same math, boundary and partial-gradient format as train_fwd_bwd2_kernel (derivation in the header of train.cu;
// reference: /root/reference/spock_reg_model.py:486-528,547-593,722-732).  What changed, and why (ncu of v2:
// shared-memory scoreboard stalls 28 %, barrier stalls 24 %, FMAs only 41 % of the executed instructions):
// The kernel is bound by shared-memory wavefronts, not FMA issue: an LDS.128 costs four wavefronts (one per quarter
// warp, 128 B each, no broadcast across quarters -- ncu: "ideal" = 4 per instruction), i.e. shared memory fills 32
// register words per cycle per SM against 128 FMA lanes, so a thread needs >= 4 FMAs per loaded word.
//   * row GEMMs (feature_nn forward, the two activation-gradient GEMMs, g_x): 4 rows x 8 columns per thread
//     (3 LDS.128 per 16 FFMA2 = 2.7 FMA per word) instead of 4 x 4 (2.0); thread = (column group, row quad) with the
//     quad fastest, so a quarter warp reads 8 consecutive 16-byte chunks of activations and ONE weight address, and
//     its epilogue STS.128 are conflict-free (quad-slowest ordering cost 2x on weight loads, 5x on the stores);
//   * weight-gradient outer products: warp-level tensor-core tiles (mma.sync.m16n8k8 tf32, 3xTF32 split in registers,
//     two passes with <= 36 live accumulators per thread, the accumulators of the other pass stashed in TENSOR MEMORY --
//     80 columns per thread, used as a register spill area, not as an MMA accumulator); 8 x 8 FFMA blocks per thread
//     (16 LDS.128 per 256 FFMA) were the round-1 first version;
//   * the Philox input noise of the next tiles is drawn by FOUR DEDICATED PRODUCER WARPS, up to two tiles ahead, into an
//     L2-resident scratch (x' and x' - mask(x), feature-major; named barriers ready / free per scratch parity), so the
//     twelve pipeline warps never wait for noise; the load phase is a float4 copy (it was 19 % of the kernel when every
//     thread drew noise between two barriers);
//   * regress_nn weights live in shared memory (six L2-latency-bound mat-vec phases per pair of systems before);
//   * the head's weight gradients are rank-1 updates per system: the vectors they need go to a 1 kB record per
//     system in the workspace and the outer products run once, at the end of the kernel, over the CTA's records --
//     no head accumulators live through the main loop;
//   * bias gradients and the 41st input column are row sums done by the two warps that have no g_x tile.
// One CTA per SM, 512 threads = 12 pipeline warps (NMAIN = 384) + 4 producer warps (NPROD = 128), 128 registers, 231.9 kB
// of shared memory, two systems (2T rows) per iteration.  Since round 2 this is the FALLBACK of bnn_train_step (batches
// below 256, flag sets whose input image does not fit the tensor-core kernel's plan) and the kernel behind bnn_saliency;
// the default training kernel is train_tc.cuh (all eight GEMMs of a system on tcgen05).
#pragma once
#include "tc.cuh"

namespace bnn {
namespace train {

constexpr int NMAIN = 384, NPROD = 128, NTHR3 = NMAIN + NPROD, HALF3 = 192;   // 12 pipeline warps + 4 producer warps
constexpr int REC = 256;     // floats per system record (head vectors for the deferred outer products)
constexpr int SMALL3 = 512;  // per-system-slot scratch (floats)
constexpr int XSM = 192;    // per-parity small inputs in the tile scratch: 2 slots x (eps12[40] eps_sum[40] y[2] pad)
constexpr int W0NP = 44;     // pitch of the natural-layout W0 rows (g_x GEMM reads 48 columns; the tail is discarded)

// per-slot scratch layout (floats); [V3_REC0, V3_REC0 + 242) is copied verbatim into the system's record
enum { V3_M = 0, V3_VAR = 20, V3_SIM = 40, V3_SIV = 60, V3_VS = 80, V3_S = 100, V3_GS = 140, V3_GM = 180, V3_GV = 200,
       V3_E12 = 220, V3_ESN = 260, V3_Y = 300,
       V3_REC0 = 304, V3_SP = 304, V3_R1 = 344, V3_R2 = 384, V3_G1 = 424, V3_G2 = 464 };
// record layout: s'[40] r1[40] r2[40] g_a1[40] g_a2[40] | dlvs[40] g_r[2] live right behind G2 in the record only
enum { R_SP = 0, R_R1 = 40, R_R2 = 80, R_G1 = 120, R_G2 = 160, R_DLVS = 200, R_GR = 240 };
// shared constants (floats, one copy)
enum { C3_ELVH = 0, C3_LVS = 40, C3_NSC = 80, C3_KLC = 144 /* exp(lv) - lv - 1 */, C3_TOTAL = 184 };

struct Smem3 {
    int RP, xT, h1T, h2T, fT, g2T, g1T, W0T, b0, W1T, b1, W2T, b2, W2n, W1n, W0n, V0, V1, V2, cb, consts, small, prod, total;
    __host__ __device__ Smem3(int T, int F) {
        RP = 2 * T + 4;
        int o = 0;
        xT = o; o += F * RP;
        h1T = o; o += H * RP;
        h2T = o; o += H * RP;
        fT = o; o += L * RP;
        g2T = o; o += H * RP;
        g1T = o; o += H * RP;
        W0T = o; o += F * H;
        b0 = o; o += H;
        W1T = o; o += H * H;
        b1 = o; o += H;
        W2T = o; o += H * L;
        b2 = o; o += L;
        W2n = o; o += L * H;
        W1n = o; o += H * H;
        W0n = o; o += H * W0NP;
        V0 = o; o += H * S2;
        V1 = o; o += H * H;
        V2 = o; o += 2 * H;
        cb = o; o += 2 * H + 4;   // c0[40] c1[40] c2[2]
        consts = o; o += C3_TOTAL;
        small = o; o += 2 * SMALL3;
        prod = o; o += 2 * 32;    // ProdArgs of the tiles being produced (by parity), TMEM base in the last word
        total = o;
    }
};

#ifdef BNN_TRAIN_TIMELINE
constexpr int TL_N = 24;
__device__ unsigned long long g_train_tl[TL_N];
// volatile + memory clobber: the read stays on its side of the neighbouring barrier
__device__ __forceinline__ long long tl_clock() {
    long long t;
    asm volatile("mov.u64 %0, %%clock64;" : "=l"(t) :: "memory");
    return t;
}
#define TL3(i)                                                 \
    do {                                                       \
        if (tid == 0) {                                        \
            const long long t_now_ = tl_clock();               \
            tl[i] += (unsigned long long)(t_now_ - tl_prev);   \
            tl_prev = t_now_;                                  \
        }                                                      \
    } while (0)
// producer-side stamps (thread 256): cycles inside produce call i -> slot 18 + i
#define TLP_BEGIN() const long long tp0_ = tl_clock()
#define TLP_END(i) do { const long long tp1_ = tl_clock(); if (tid == NMAIN) tl[18 + (i)] += (unsigned long long)(tp1_ - tp0_); } while (0)
#else
#define TL3(i) do { } while (0)
#define TLP_BEGIN() do { } while (0)
#define TLP_END(i) do { } while (0)
#endif

// acc2[r][i] (columns c0 + 2i, c0 + 2i + 1 of row 4q + r) += sum_k AT[k][4q + r] * W[k][c0 + 2i .. +1]
template <int RP, int K, int NP, int NC>
__device__ __forceinline__ void rowgemm4(const float* __restrict__ AT, const float* __restrict__ W, int q, int c0,
                                         u64 (&a2)[4][NC / 2]) {
    const float* ap = AT + 4 * q;
    const float* wp = W + c0;
#pragma unroll 4
    for (int k = 0; k < K; ++k) {
        const float4 a = *reinterpret_cast<const float4*>(ap + k * RP);
        u64 w[NC / 2];
#pragma unroll
        for (int i = 0; i < NC / 4; ++i) {
            const ulonglong2 t = *reinterpret_cast<const ulonglong2*>(wp + k * NP + 4 * i);
            w[2 * i] = t.x;
            w[2 * i + 1] = t.y;
        }
        const u64 av[4] = {pack2(a.x, a.x), pack2(a.y, a.y), pack2(a.z, a.z), pack2(a.w, a.w)};
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int i = 0; i < NC / 2; ++i) a2[r][i] = fma2(av[r], w[i], a2[r][i]);
    }
}

// outer-product variant: 16 = warp-level tensor-core tiles (mma.sync 3xTF32, default), 48 = 4 x 8 FFMA2 blocks,
// 88 = 8 x 8 FFMA blocks
#ifndef V3_OUTER
#define V3_OUTER 16
#endif
// 4 x 8 variant: even / odd rows accumulate in the two halves of an fp32x2 register (no packing moves)
__device__ __forceinline__ void outer4x8(const float* __restrict__ Gp, int gstr, const float* __restrict__ Hp, int hstr,
                                         int q0, int q1, float (&acc)[4][8]) {
    u64 a2[4][8];
#pragma unroll
    for (int jj = 0; jj < 4; ++jj)
#pragma unroll
        for (int kk = 0; kk < 8; ++kk) a2[jj][kk] = pack2(acc[jj][kk], 0.f);
#pragma unroll 1
    for (int q = q0; q < q1; ++q) {
        ulonglong2 g[4];
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) g[jj] = *reinterpret_cast<const ulonglong2*>(Gp + jj * gstr + 4 * q);
#pragma unroll
        for (int kk = 0; kk < 8; ++kk) {
            const ulonglong2 h = *reinterpret_cast<const ulonglong2*>(Hp + kk * hstr + 4 * q);
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) {
                a2[jj][kk] = fma2(g[jj].x, h.x, a2[jj][kk]);
                a2[jj][kk] = fma2(g[jj].y, h.y, a2[jj][kk]);
            }
        }
    }
#pragma unroll
    for (int jj = 0; jj < 4; ++jj)
#pragma unroll
        for (int kk = 0; kk < 8; ++kk) {
            float lo, hi;
            unpack2(a2[jj][kk], lo, hi);
            acc[jj][kk] = lo + hi;
        }
}

// acc[jj][kk] += sum over the rows of quads [q0, q1) of G[jj * gstr][r] * Hm[kk * hstr][r]  (feature-major, pitch RP)
__device__ __forceinline__ void outer8x8(const float* __restrict__ Gp, int gstr, const float* __restrict__ Hp, int hstr,
                                         int q0, int q1, float (&acc)[8][8]) {
#pragma unroll 1
    for (int q = q0; q < q1; ++q) {
        float4 g[8];
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) g[jj] = *reinterpret_cast<const float4*>(Gp + jj * gstr + 4 * q);
#pragma unroll
        for (int kk = 0; kk < 8; ++kk) {
            const float4 h = *reinterpret_cast<const float4*>(Hp + kk * hstr + 4 * q);
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) {
                float a = acc[jj][kk];
                a = fmaf(g[jj].x, h.x, a);
                a = fmaf(g[jj].y, h.y, a);
                a = fmaf(g[jj].z, h.z, a);
                a = fmaf(g[jj].w, h.w, a);
                acc[jj][kk] = a;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Warp-level tensor-core tiles: mma.sync.m16n8k8, tf32 x tf32 -> fp32, operands in registers (512 MAC per cycle per SM
// measured, tools/mma_sync_rate.py: 4 x the FP32 FMA rate).  Full fp32 accuracy comes from the 3xTF32 split done in
// registers (hi = cvt.rna.tf32, lo = x - hi; lo.hi + hi.lo first, hi.hi last), so that three MMAs = one fp32-grade
// 16 x 8 x 8 tile: 1.33 x the FP32 roofline, with 22 LDS.32 per 15 tiles instead of 12 LDS.128 per 4 x 8 x 4 block.
// Fragment layout (g = lane / 4, t = lane % 4): A a0 = (g, t) a1 = (g+8, t) a2 = (g, t+4) a3 = (g+8, t+4);
// B b0 = (k = t, n = g) b1 = (t+4, g); D c0 = (g, 2t) c1 = (g, 2t+1) c2 = (g+8, 2t) c3 = (g+8, 2t+1).
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mma_tf32(float (&c)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
    asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}
__device__ __forceinline__ void split_tf32(float x, uint32_t& hi, uint32_t& lo) {
    // round to nearest on the 13 dropped mantissa bits with two integer ops (cvt.rna.tf32 goes through the
    // conversion unit at a fraction of the ALU rate and was as expensive as the MMAs it feeds)
    hi = (__float_as_uint(x) + 0x1000u) & 0xffffe000u;
    lo = __float_as_uint(x - __uint_as_float(hi));
}

// acc[nt][4 mt + i] (16 x 8 tiles of D[m][n], three row tiles mt per column tile nt; 16 stash columns per nt, 12 used)
// += sum over the rows of k-steps [ks0, ks1) (8 rows each) of Ms[(16 mt + m)][r] * Ns[(8 nt + n)][r]; both operands
// feature-major with pitch RP: dW[j = n][k = m] of one layer.  RP = 12 mod 32 makes every fragment LDS.32 one
// conflict-free wavefront (bank = 12 g + t).  NN column tiles per call: 36 accumulators in registers at most.
template <int RP, int NN>
__device__ __forceinline__ void outer_mma(const float* __restrict__ Ms, const float* __restrict__ Ns, int ks0, int ks1,
                                          int lane, float (&acc)[NN][16]) {
    const int g = lane >> 2, t = lane & 3;
    const float* mp = Ms + g * RP + t;
    const float* np_ = Ns + g * RP + t;
#pragma unroll 1
    for (int ks = ks0; ks < ks1; ++ks) {
        const int r0 = 8 * ks;
        uint32_t ah[3][4], al[3][4];
#pragma unroll
        for (int mt = 0; mt < 3; ++mt) {
            const float* p = mp + 16 * mt * RP + r0;
            split_tf32(p[0], ah[mt][0], al[mt][0]);
            split_tf32(p[8 * RP], ah[mt][1], al[mt][1]);
            split_tf32(p[4], ah[mt][2], al[mt][2]);
            split_tf32(p[8 * RP + 4], ah[mt][3], al[mt][3]);
        }
        uint32_t bh[NN][2], bl[NN][2];
#pragma unroll
        for (int nt = 0; nt < NN; ++nt) {
            const float* p = np_ + 8 * nt * RP + r0;
            split_tf32(p[0], bh[nt][0], bl[nt][0]);
            split_tf32(p[4], bh[nt][1], bl[nt][1]);
        }
        // three passes over the 3 NN independent tiles: consecutive MMAs never touch the same accumulator
#pragma unroll
        for (int pass = 0; pass < 3; ++pass)
#pragma unroll
            for (int nt = 0; nt < NN; ++nt)
#pragma unroll
                for (int mt = 0; mt < 3; ++mt) {
                    float (&c)[4] = *reinterpret_cast<float (*)[4]>(&acc[nt][4 * mt]);
                    if (pass == 0) mma_tf32(c, al[mt], bh[nt]);
                    else if (pass == 1) mma_tf32(c, ah[mt], bl[nt]);
                    else mma_tf32(c, ah[mt], bh[nt]);
                }
    }
}

// Row GEMM on the same tiles: C[row][n] = sum_k AT[k][row] * W[k][n] over the 2T = 200 rows (12 full 16-row tiles +
// one half-used tile), K padded to a multiple of 8 with zero operands, N = 8 * NNT columns (pad columns read whatever
// follows W and are dropped by the epilogue).  Warp w owns rows [16 w, 16 w + 16) with all NNT column tiles (its A
// fragments are loaded and split once per k-step) and, for w < NNT, the tile (rows 192.., columns 8 w..) of the 13th
// row tile (accx).  The caller runs the epilogue over acc[nt] (rows 16 w + g (+8), columns 8 nt + 2 t (+1)) and accx.
// V3_GEMM: 0 = the six row GEMMs on 4 x 8 FFMA2 register tiles (default), 1 = on the same mma.sync tiles as the outer
// products.  Measured (4 seeds x 2000): 0.754 ms vs 1.115 ms per step -- for the row GEMMs the 3xTF32 tile rate of the
// legacy tensor path (three 8-cycle MMAs per 16 x 8 x 8 = 1.33 x the FP32 FMA rate, 0.85 of it left after padding
// 200 x 41 / 20 to tile multiples) does not beat FFMA2 tiles that already run from registers, and every layer pays
// two splits per operand word; the outer products win because their operand traffic drops 8-fold.  Also tried for the row
// GEMMs: 8 rows x 8 columns per thread (4.0 FMA per loaded word instead of 2.7; 125 threads = one warp per scheduler):
// 0.91 ms -- a single warp per scheduler cannot cover its own LDS latency.
#ifndef V3_GEMM
#define V3_GEMM 0
#endif
template <int RP, int K, int NP, int NNT>
__device__ __forceinline__ void rowgemm_mma(const float* __restrict__ AT, const float* __restrict__ W, int warp, int lane,
                                            float (&acc)[NNT][4], float (&accx)[4]) {
    const int g = lane >> 2, t = lane & 3;
    constexpr int KS = (K + 7) / 8;
    constexpr bool KPAD = (K % 8) != 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) accx[i] = 0.f;
#pragma unroll
    for (int nt = 0; nt < NNT; ++nt)
#pragma unroll
        for (int i = 0; i < 4; ++i) acc[nt][i] = 0.f;
    const bool has_x = warp < NNT;
    const float* ap = AT + t * RP + 16 * warp + g;
    const float* axp = AT + t * RP + 192 + g;
    const float* wp = W + t * NP + g;
#pragma unroll 1
    for (int ks = 0; ks < KS; ++ks) {
        const int k0 = 8 * ks;
        const bool v0 = !KPAD || (k0 + t < K), v1 = !KPAD || (k0 + t + 4 < K);
        uint32_t ah[4], al[4], xh[4], xl[4];
        split_tf32(v0 ? ap[k0 * RP] : 0.f, ah[0], al[0]);
        split_tf32(v0 ? ap[k0 * RP + 8] : 0.f, ah[1], al[1]);
        split_tf32(v1 ? ap[(k0 + 4) * RP] : 0.f, ah[2], al[2]);
        split_tf32(v1 ? ap[(k0 + 4) * RP + 8] : 0.f, ah[3], al[3]);
        if (has_x) {
            split_tf32(v0 ? axp[k0 * RP] : 0.f, xh[0], xl[0]);
            split_tf32(v0 ? axp[k0 * RP + 8] : 0.f, xh[1], xl[1]);
            split_tf32(v1 ? axp[(k0 + 4) * RP] : 0.f, xh[2], xl[2]);
            split_tf32(v1 ? axp[(k0 + 4) * RP + 8] : 0.f, xh[3], xl[3]);
        }
        uint32_t bh[NNT][2], bl[NNT][2];
#pragma unroll
        for (int nt = 0; nt < NNT; ++nt) {
            split_tf32(v0 ? wp[k0 * NP + 8 * nt] : 0.f, bh[nt][0], bl[nt][0]);
            split_tf32(v1 ? wp[(k0 + 4) * NP + 8 * nt] : 0.f, bh[nt][1], bl[nt][1]);
        }
        // three passes over the independent tiles: consecutive MMAs never touch the same accumulator
#pragma unroll
        for (int pass = 0; pass < 3; ++pass) {
#pragma unroll
            for (int nt = 0; nt < NNT; ++nt) {
                if (pass == 0) mma_tf32(acc[nt], al, bh[nt]);
                else if (pass == 1) mma_tf32(acc[nt], ah, bl[nt]);
                else mma_tf32(acc[nt], ah, bh[nt]);
                if (has_x && nt == warp) {
                    if (pass == 0) mma_tf32(accx, xl, bh[nt]);
                    else if (pass == 1) mma_tf32(accx, xh, bl[nt]);
                    else mma_tf32(accx, xh, bh[nt]);
                }
            }
        }
    }
}
// epilogues of one tile: c0 = (row, col), c1 = (row, col + 1), c2 = (row + 8, col), c3 = (row + 8, col + 1); full = rows + 8 exist
template <int RP, bool RELU>
__device__ __forceinline__ void tile_store_bias(float* __restrict__ out, const float* __restrict__ bias, int row, int col,
                                                const float (&c)[4], bool full) {
    const float bA = bias[col], bB = bias[col + 1];
    float v0 = c[0] + bA, v1 = c[1] + bB, v2 = c[2] + bA, v3 = c[3] + bB;
    if (RELU) { v0 = relu_nan(v0); v1 = relu_nan(v1); v2 = relu_nan(v2); v3 = relu_nan(v3); }
    out[col * RP + row] = v0;
    out[(col + 1) * RP + row] = v1;
    if (full) { out[col * RP + row + 8] = v2; out[(col + 1) * RP + row + 8] = v3; }
}
template <int RP>
__device__ __forceinline__ void tile_store_masked(float* __restrict__ out, const float* __restrict__ hT, int row, int col,
                                                  const float (&c)[4], bool full) {
    out[col * RP + row] = hT[col * RP + row] > 0.f ? c[0] : 0.f;
    out[(col + 1) * RP + row] = hT[(col + 1) * RP + row] > 0.f ? c[1] : 0.f;
    if (full) {
        out[col * RP + row + 8] = hT[col * RP + row + 8] > 0.f ? c[2] : 0.f;
        out[(col + 1) * RP + row + 8] = hT[(col + 1) * RP + row + 8] > 0.f ? c[3] : 0.f;
    }
}

// Tensor memory as a register stash: a thread's block of weight-gradient accumulators lives in its own TMEM lane
// (columns [col, col + NV)) between the outer-product phases, so that no other phase carries those registers.
template <int NV>
__device__ __forceinline__ void stash_load(uint32_t taddr, float* v) {
#pragma unroll
    for (int i = 0; i < NV / 16; ++i) {
        uint32_t u[16];
        tmem_ld16(taddr + 16 * i, u);
        tc_wait_ld();
#pragma unroll
        for (int j = 0; j < 16; ++j) v[16 * i + j] = __uint_as_float(u[j]);
    }
}
template <int NV>
__device__ __forceinline__ void stash_store(uint32_t taddr, const float* v) {
#pragma unroll
    for (int i = 0; i < NV / 16; ++i) {
        uint32_t u[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) u[j] = __float_as_uint(v[16 * i + j]);
        tmem_st16(taddr + 16 * i, u);
    }
    tc_wait_st();
}

// Input tile producer: x' = mask(x) + eps_in * exp(lv_in / 2) (:486-500) and n = x' - mask(x) for the two systems
// b0n, b0n + 1 (data rows row0 / row1, -1 = past the batch), written feature-major ([c][2T]) to this CTA's scratch.
// Work items are (system slot, 4-column group, time step); item ids first + stride * round, round in [r0, r0 + NR).
// All loads of the NR rounds are issued before the first Philox block (the rounds were latency-bound one by one).
// Philox counters as in train_noise_kernel.  Not inlined: six call sites, ~500 instructions each.
struct ProdArgs {
    const float* X; const float* eps_in; float* xp; float* np; const float* nsc;
    const float* Y; const float* eps12; const float* eps_sum; float* sm_out;
    uint64_t key, zero_mask; int64_t sb0; int row0, row1, b0n, step, saliency;
};
static_assert(sizeof(ProdArgs) <= 31 * sizeof(float), "ProdArgs must fit its shared-memory slot");
template <int T, int F, int NR>
__device__ __noinline__ void produce_tile(const ProdArgs* __restrict__ ap, int first, int stride, int r0) {
    const ProdArgs a = *ap;
    constexpr int F4 = (F + 3) >> 2, RT = 2 * T, PER = T * F4;
    float xv[NR][4], ev[NR][4];
    int off[NR], c4s[NR];
    uint4 ctr[NR];
    bool live[NR];
    // straight-line loads: out-of-range items / columns are clamped to a valid address and masked at the store
#pragma unroll
    for (int k = 0; k < NR; ++k) {
        const int id0 = first + stride * (r0 + k);
        const bool ok = id0 < 2 * PER;
        const int id = ok ? id0 : 2 * PER - 1;
        const int hs = id >= PER ? 1 : 0, rem = id - hs * PER;
        const int c4 = rem / T, t = rem - c4 * T;
        const int row = hs ? a.row1 : a.row0;
        c4s[k] = c4;
        off[k] = ok ? hs * T + t : -1;
        live[k] = row >= 0;
        ctr[k] = make_uint4((uint32_t)(t * F4 + c4), (uint32_t)(a.b0n + hs), (uint32_t)a.step, STREAM_EPS_IN);
        const float* xs = a.X + ((int64_t)(row >= 0 ? row : 0) * T + t) * F;
#pragma unroll
        for (int u = 0; u < 4; ++u) xv[k][u] = __ldg(xs + min(4 * c4 + u, F - 1));
    }
    if (a.eps_in && !a.saliency) {
#pragma unroll
        for (int k = 0; k < NR; ++k) {
            const int t = (int)ctr[k].x / F4, hs = (int)ctr[k].y - a.b0n;
            const float* es = a.eps_in + ((a.sb0 + (live[k] ? hs : 0)) * T + t) * (int64_t)F;
#pragma unroll
            for (int u = 0; u < 4; ++u) ev[k][u] = __ldg(es + min(4 * c4s[k] + u, F - 1));
        }
    }
    if (a.saliency) {   // noise-free input (feature_importance.py: gradforward has no input noise)
#pragma unroll
        for (int k = 0; k < NR; ++k)
#pragma unroll
            for (int u = 0; u < 4; ++u) ev[k][u] = 0.f;
    } else if (!a.eps_in) {
        // NR Philox4x32-10 blocks, rounds interleaved across the blocks (one warp per scheduler runs this: the
        // instruction-level parallelism has to come from here)
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
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int c = 4 * c4s[k] + u;
            if (c < F && off[k] >= 0) {
                float x = xv[k][u];
                if ((a.zero_mask >> c) & 1ull) x = __fsub_rn(x, x);  // x - mask keeps NaN (:452-478)
                const float xpv = live[k] ? __fadd_rn(x, __fmul_rn(ev[k][u], a.nsc[c])) : 0.f;
                a.xp[c * RT + off[k]] = xpv;
                a.np[c * RT + off[k]] = live[k] ? __fsub_rn(xpv, x) : 0.f;
            }
        }
    }
}

// The per-system vectors of the same tile: eps1|eps2 (:426-427), the summary noise (:522) and the labels, for both slots.
// Threads p < 20 (two slots x 10 float4) draw / load the noise, p = 32, 33 fetch the labels.
__device__ __noinline__ void produce_small(const ProdArgs* __restrict__ ap, int p) {
    const ProdArgs a = *ap;
    if (p < 20) {
        const int hs = p / 10, l = p - 10 * hs;
        const int row = hs ? a.row1 : a.row0;
        float4 e = make_float4(0.f, 0.f, 0.f, 0.f), c = e;
        if (row >= 0) {
            if (a.eps12) {
                e = __ldg(reinterpret_cast<const float4*>(a.eps12 + (a.sb0 + hs) * S2) + l);
                if (a.eps_sum) c = __ldg(reinterpret_cast<const float4*>(a.eps_sum + (a.sb0 + hs) * S2) + l);
            } else {
                e = philox_normal4(a.key, STREAM_EPS, (uint32_t)(a.b0n + hs), (uint32_t)a.step, (uint32_t)l);
                c = philox_normal4(a.key, STREAM_EPS_SUM, (uint32_t)(a.b0n + hs), (uint32_t)a.step, (uint32_t)l);
            }
            if (a.saliency) c = make_float4(0.f, 0.f, 0.f, 0.f);   // partforward adds no summary noise
        }
        reinterpret_cast<float4*>(a.sm_out + hs * (XSM / 2))[l] = e;
        reinterpret_cast<float4*>(a.sm_out + hs * (XSM / 2) + S2)[l] = c;
    } else if (p == 32 || p == 33) {
        const int hs = p - 32;
        const int row = hs ? a.row1 : a.row0;
        float2 y = make_float2(0.f, 0.f);
        if (row >= 0 && a.Y) y = __ldg(reinterpret_cast<const float2*>(a.Y) + row);
        *reinterpret_cast<float2*>(a.sm_out + hs * (XSM / 2) + 2 * S2) = y;
    }
}

// Named barriers.  0: whole CTA (prologue only); 1, 2: tile of parity 0 / 1 is ready (producers arrive, pipeline waits);
// 3, 4: scratch of parity 0 / 1 is free again (pipeline arrives, producers wait); 5: the 12 pipeline warps; 6: the producers.
__device__ __forceinline__ void nb_sync(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ void nb_arrive(int id, int n) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(n) : "memory"); }
#define MAIN_SYNC() nb_sync(5, NMAIN)

template <int T, int F>
__global__ void __launch_bounds__(NTHR3, 1) train_fwd_bwd3_kernel(const Params prm) {
    extern __shared__ __align__(16) float sm[];
    constexpr int NQ = T >> 2, NQ2 = 2 * NQ, RT = 2 * T, RP = 2 * T + 4;
    static_assert(F == 41 && T == 100, "thread maps below are laid out for the reference's shape");
    const Smem3 L_(T, F);
    const FlatLayout fl(F);
    const int tid = threadIdx.x;
    const int half = tid >= HALF3 ? 1 : 0, lt = tid - half * HALF3;
    const int lane = tid & 31;
    const int sidx = prm.seed0 + (int)blockIdx.y;
    const float* th = prm.theta + (int64_t)sidx * fl.d;
    float* xT = sm + L_.xT; float* h1T = sm + L_.h1T; float* h2T = sm + L_.h2T; float* fT = sm + L_.fT;
    float* g2T = sm + L_.g2T; float* g1T = sm + L_.g1T;
    float* W0T = sm + L_.W0T; float* b0 = sm + L_.b0; float* W1T = sm + L_.W1T; float* b1 = sm + L_.b1;
    float* W2T = sm + L_.W2T; float* b2 = sm + L_.b2; float* W2n = sm + L_.W2n; float* W1n = sm + L_.W1n; float* W0n = sm + L_.W0n;
    float* V0s = sm + L_.V0; float* V1s = sm + L_.V1; float* V2s = sm + L_.V2; float* cbs = sm + L_.cb;
    float* cst = sm + L_.consts;
    float* sv = sm + L_.small + half * SMALL3;
#ifdef BNN_TRAIN_TIMELINE
    unsigned long long tl[TL_N];
#pragma unroll
    for (int i = 0; i < TL_N; ++i) tl[i] = 0;
    long long tl_prev = tl_clock();
#endif

    // ---- stage this seed's weights (feature matrices natural and transposed, the head natural) ----
    for (int i = tid; i < H * F; i += NTHR3) {
        const int j = i / F, c = i - j * F;
        const float w = __ldg(th + fl.W0 + i);
        W0T[c * H + j] = w;
        W0n[j * W0NP + c] = w;
    }
    for (int i = tid; i < H * (W0NP - F); i += NTHR3) W0n[(i / (W0NP - F)) * W0NP + F + i % (W0NP - F)] = 0.f;
    for (int i = tid; i < H * H; i += NTHR3) {
        const int j = i / H, k = i - j * H;
        const float w = __ldg(th + fl.W1 + i);
        W1T[k * H + j] = w;
        W1n[i] = w;
        V1s[i] = __ldg(th + fl.V1 + i);
        V0s[i] = __ldg(th + fl.V0 + i);   // H * S2 == H * H
    }
    for (int i = tid; i < L * H; i += NTHR3) {
        const int j = i / H, k = i - j * H;
        const float w = __ldg(th + fl.W2 + i);
        W2T[k * L + j] = w;
        W2n[i] = w;
    }
    if (tid < H) {
        b0[tid] = __ldg(th + fl.b0 + tid); b1[tid] = __ldg(th + fl.b1 + tid);
        cbs[tid] = __ldg(th + fl.c0 + tid); cbs[H + tid] = __ldg(th + fl.c1 + tid);
    }
    if (tid < 2 * H) V2s[tid] = __ldg(th + fl.V2 + tid);
    if (tid < 2) cbs[2 * H + tid] = __ldg(th + fl.c2 + tid);
    if (tid < L) b2[tid] = __ldg(th + fl.b2 + tid);
    if (tid < S2) {
        const float lv = __ldg(th + fl.lv_sum + tid);
        cst[C3_LVS + tid] = lv;
        cst[C3_ELVH + tid] = expf(__fdiv_rn(lv, 2.0f));
        cst[C3_KLC + tid] = expf(lv) - lv - 1.0f;   // the parameter part of the summary KL term (:515-520)
    }
    if (tid < F) cst[C3_NSC + tid] = expf(__fdiv_rn(__ldg(th + fl.lv_in + tid), 2.0f));
    // the 4 pad rows of every feature row are never read (row GEMMs and outer products stop at 2T)

    // ---- thread roles ----
    // row GEMMs: column group cg_rg (8 columns; 4 for the latent layer), quad q_rg of the 2T rows, quad fastest
    const int cg_rg = tid / NQ2, q_rg = tid - NQ2 * cg_rg;   // 5 groups: tid < 250; g_x (48 columns, 6 groups): tid < 300
    // outer products: one block of one matrix over one row group
    const float* opG; const float* opH; int op_gstr, op_q0, op_q1, op_role, op_jb, op_kb;
#if V3_OUTER == 16
    // warp-level tensor-core tiles: warps 0..4 dW0 (M side x', 48 x 40), 5..9 dW1 (h1, 48 x 40), five k-steps of 8 rows
    // each; warps 10, 11 dW2 (h2 x g_f, 48 x 24), 13 / 12 k-steps.  60 accumulators per thread (36 for dW2).
    const int owarp = tid >> 5;
    op_role = owarp < 5 ? 0 : (owarp < 10 ? 1 : 2);
    opG = op_role == 0 ? g1T : (op_role == 1 ? g2T : fT);    // N side (output index j)
    opH = op_role == 0 ? xT : (op_role == 1 ? h1T : h2T);    // M side (input index k)
    op_q0 = op_role == 0 ? 5 * owarp : (op_role == 1 ? 5 * (owarp - 5) : (owarp == 10 ? 0 : 13));
    op_q1 = op_role == 0 ? 5 * owarp + 5 : (op_role == 1 ? 5 * (owarp - 5) + 5 : (owarp == 10 ? 13 : 25));
    op_gstr = 0; op_jb = 0; op_kb = 0;
    constexpr int OJ = 10;   // 80 stash columns per thread: 5 column tiles x 16 (12 used)
#elif V3_OUTER == 88
    // 8 x 8 blocks, six row groups (dW2: five)
    {
        int r = tid, rg;
        if (tid < 150) { op_role = 0; rg = r / 25; r -= 25 * rg; opG = g1T; opH = xT; }
        else if (tid < 300) { op_role = 1; r -= 150; rg = r / 25; r -= 25 * rg; opG = g2T; opH = h1T; }
        else if (tid < 375) { op_role = 2; r -= 300; rg = r / 15; r -= 15 * rg; opG = fT; opH = h2T; }
        else { op_role = 3; rg = 0; r = 0; opG = fT; opH = h2T; }
        op_jb = r / 5; op_kb = r - 5 * op_jb;
        op_gstr = (op_role >= 2 ? 3 : 5) * RP;   // dW2: rows j = jb + 3 jj (j >= 20 is discarded), else j = jb + 5 jj
        opG += op_jb * RP; opH += op_kb * RP;
        if (op_role < 2) { op_q0 = rg < 2 ? 9 * rg : 18 + 8 * (rg - 2); op_q1 = rg < 2 ? 9 * rg + 9 : 26 + 8 * (rg - 2); }
        else if (op_role == 2) { op_q0 = 10 * rg; op_q1 = 10 * rg + 10; }
        else { op_q0 = 0; op_q1 = 0; }
    }
    constexpr int OJ = 8;
#else
    // 4 x 8 blocks (fp32x2 accumulators), three row groups
    {
        int r = tid, rg;
        if (tid < 150) { op_role = 0; rg = r / 50; r -= 50 * rg; op_jb = r / 5; op_kb = r - 5 * op_jb; opG = g1T; opH = xT; op_gstr = 10 * RP; }
        else if (tid < 300) { op_role = 1; r -= 150; rg = r / 50; r -= 50 * rg; op_jb = r / 5; op_kb = r - 5 * op_jb; opG = g2T; opH = h1T; op_gstr = 10 * RP; }
        else if (tid < 375) { op_role = 2; r -= 300; rg = r / 25; r -= 25 * rg; op_jb = r / 5; op_kb = r - 5 * op_jb; opG = fT; opH = h2T; op_gstr = 5 * RP; }
        else { op_role = 3; rg = 0; op_jb = 0; op_kb = 0; opG = fT; opH = h2T; op_gstr = 5 * RP; }
        opG += op_jb * RP; opH += op_kb * RP;
        op_q0 = rg == 0 ? 0 : (rg == 1 ? 17 : 34);
        op_q1 = op_role == 3 ? 0 : (rg == 0 ? 17 : (rg == 1 ? 34 : NQ2));
    }
    constexpr int OJ = 4;
#endif
    // the block's accumulators: OJ * 8 columns of this thread's TMEM lane (three warps share a lane quadrant)
#if V3_GEMM == 1
    constexpr int NV = OJ * 8, TSTRIDE = NV + 16, TCOLS = 512;   // + 16 columns per thread for the dlv_in partial sums
#else
    constexpr int NV = OJ * 8, TSTRIDE = NV, TCOLS = NV == 32 ? 128 : 256;   // three warps per lane quadrant: 3 NV <= TCOLS
#endif
    uint32_t* tslot = reinterpret_cast<uint32_t*>(sm + L_.prod + 63);
    if (tid < 32) { tmem_alloc(tslot, TCOLS); tmem_relinquish(); }
    tc_fence_before();
    __syncthreads();   // whole CTA: weights, noise scales and the TMEM base are staged
    tc_fence_after();
    const uint32_t tbase = *tslot;
    const uint64_t key = seed_key(prm.seed, sidx);
    // this CTA's input-tile scratch: [parity][x' | n | small inputs]
    constexpr int XPAR = 2 * F * RT + XSM;
    float* xprod = prm.xprod + ((int64_t)sidx * prm.n_cta + blockIdx.x) * (2 * XPAR);

    // =====================================================================================================
    // Producer warps (12..15): run up to two tiles ahead of the pipeline, never touch its barriers.
    // =====================================================================================================
    if (tid >= NMAIN) {
        const int ptid = tid - NMAIN;
#ifdef BNN_TRAIN_TIMELINE
        long long tp_wait = 0, tp_work = 0;
#endif
        int it = 0;
        for (int b0p = 2 * blockIdx.x; b0p < prm.B; b0p += 2 * gridDim.x, ++it) {
            const int par = it & 1;
#ifdef BNN_TRAIN_TIMELINE
            const long long t0 = tl_clock();
#endif
            if (it >= 2) nb_sync(3 + par, NTHR3);   // the pipeline is done with the tile that used this parity
#ifdef BNN_TRAIN_TIMELINE
            const long long t1 = tl_clock();
#endif
            ProdArgs* pas = reinterpret_cast<ProdArgs*>(sm + L_.prod) + par;
            float* xo = xprod + par * XPAR;
            if (ptid == 0) {
                const int64_t sbq = (int64_t)sidx * prm.B + b0p;
                pas->X = prm.X; pas->eps_in = prm.eps_in; pas->nsc = cst + C3_NSC; pas->key = key; pas->zero_mask = prm.zero_mask;
                pas->step = (int)prm.step; pas->Y = prm.Y; pas->eps12 = prm.eps12; pas->eps_sum = prm.eps_sum;
                pas->saliency = prm.saliency;
                pas->b0n = b0p; pas->sb0 = sbq; pas->xp = xo; pas->np = xo + F * RT; pas->sm_out = xo + 2 * F * RT;
                pas->row0 = prm.batch_index ? prm.batch_index[sbq] : b0p;
                pas->row1 = b0p + 1 < prm.B ? (prm.batch_index ? prm.batch_index[sbq + 1] : b0p + 1) : -1;
            }
            {   // pull the rows of the next tile into L2
                const int b2n = b0p + 2 * gridDim.x;
                constexpr int LINES = (T * F * 4 + 127) / 128;   // 129 lines of 128 B per system
                for (int i = ptid; i < 2 * LINES; i += NPROD) {
                    const int hs = i >= LINES ? 1 : 0, ln = i - hs * LINES;
                    if (b2n + hs < prm.B) {
                        const int64_t sb2 = (int64_t)sidx * prm.B + b2n + hs;
                        const int64_t r2 = prm.batch_index ? (int64_t)prm.batch_index[sb2] : (int64_t)(b2n + hs);
                        const char* p2 = reinterpret_cast<const char*>(prm.X + r2 * T * F) + 128 * ln;
                        asm volatile("prefetch.global.L2 [%0];" ::"l"(p2));
                    }
                }
            }
            nb_sync(6, NPROD);                       // descriptor visible to the four warps
            produce_small(pas, ptid);
            produce_tile<T, F, 6>(pas, ptid, NPROD, 0);
            produce_tile<T, F, 6>(pas, ptid, NPROD, 6);
            produce_tile<T, F, 6>(pas, ptid, NPROD, 12);
            __threadfence_block();
            nb_arrive(1 + par, NTHR3);               // tile ready
#ifdef BNN_TRAIN_TIMELINE
            tp_wait += t1 - t0; tp_work += tl_clock() - t1;
#endif
        }
#ifdef BNN_TRAIN_TIMELINE
        if (tid == NMAIN && blockIdx.x == 0 && blockIdx.y == 0) { g_train_tl[18] = tp_work; g_train_tl[19] = tp_wait; }
#endif
        return;
    }

    // =====================================================================================================
    // Pipeline warps (0..11)
    // =====================================================================================================
    const uint32_t taddr = tbase + ((uint32_t)(((tid >> 5) & 3) * 32) << 16) + (uint32_t)((tid >> 7) * TSTRIDE);
    {
        float z[NV];
#pragma unroll
        for (int i = 0; i < NV; ++i) z[i] = 0.f;
        stash_store<NV>(taddr, z);
#if V3_GEMM == 1
        stash_store<16>(taddr + NV, z);
#endif
    }
    // tid < 300: dlv_in partial sums of this thread's 8 g_x columns; tid >= 300: two of the 120 row sums
    // (rows 0..39: b0 = sum g_a1, 40..79: column 40 of dW0 = sum g_a1 x'[40], 80..119: b1 = sum g_a2)
    float aux[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#if V3_GEMM == 1
    // tensor-core row GEMMs: the dlv_in partial sums per (column tile slot, column of the pair) live in 16 stash
    // columns and are in registers only inside the g_x phase; b0 / b1 row sums (tid < 80)
    float arow = 0.f;
    (void)aux;
#endif
    float ab2 = 0.f, a_nll = 0.f, a_skl = 0.f;
    const float Tf = (float)T, Tm1 = (float)(T - 1);
    int parity = 0;
    TL3(0);

    for (int b0i = 2 * blockIdx.x; b0i < prm.B; b0i += 2 * gridDim.x) {
        const int b = b0i + half;
        const bool act = b < prm.B;
        const int64_t sb = (int64_t)sidx * prm.B + (act ? b : b0i);
        // ---- S0: copy this iteration's x' tile from the scratch (written one iteration ago by the producer warps) ----
        const float* xp_cur = xprod + parity * XPAR;
        const float* np_cur = xp_cur + F * RT;
        nb_sync(1 + parity, NTHR3);   // the producers have finished this tile
        {
            // all loads first (L2 latency once, not once per float4)
            constexpr int NCP = (F * NQ2 + NMAIN - 1) / NMAIN;
            float4 cp[NCP];
#pragma unroll
            for (int k = 0; k < NCP; ++k) {
                const int i = tid + k * NMAIN;
                cp[k] = __ldcg(reinterpret_cast<const float4*>(xp_cur) + min(i, F * NQ2 - 1));
            }
#pragma unroll
            for (int k = 0; k < NCP; ++k) {
                const int i = tid + k * NMAIN;
                if (i < F * NQ2) {
                    const int c = i / NQ2, q = i - c * NQ2;
                    *reinterpret_cast<float4*>(xT + c * RP + 4 * q) = cp[k];
                }
            }
            if (tid < 2 * 21) {   // the small inputs of both slots: eps12 | eps_sum (20 float4) and the labels
                const int hs = tid / 21, w = tid - 21 * hs;
                const float* src = xp_cur + 2 * F * RT + hs * (XSM / 2);
                float* dst = sm + L_.small + hs * SMALL3;
                if (w < 20) *reinterpret_cast<float4*>(dst + (w < 10 ? V3_E12 + 4 * w : V3_ESN + 4 * (w - 10))) =
                                __ldcg(reinterpret_cast<const float4*>(src) + w);
                else *reinterpret_cast<float2*>(dst + V3_Y) = __ldcg(reinterpret_cast<const float2*>(src + 2 * S2));
            }
        }
        MAIN_SYNC();
        TL3(1);
        // ---- S1..S3: feature_nn forward over the 2T rows ----
#if V3_GEMM == 1
        {
            const int wrp = tid >> 5, mg = lane >> 2, mt2 = 2 * (lane & 3);
            float acc[5][4], accx[4];
            rowgemm_mma<RP, F, H, 5>(xT, W0T, wrp, lane, acc, accx);
#pragma unroll
            for (int nt = 0; nt < 5; ++nt) tile_store_bias<RP, true>(h1T, b0, 16 * wrp + mg, 8 * nt + mt2, acc[nt], true);
            if (wrp < 5) tile_store_bias<RP, true>(h1T, b0, 192 + mg, 8 * wrp + mt2, accx, false);
        }
        MAIN_SYNC();
        TL3(2);
        {
            const int wrp = tid >> 5, mg = lane >> 2, mt2 = 2 * (lane & 3);
            float acc[5][4], accx[4];
            rowgemm_mma<RP, H, H, 5>(h1T, W1T, wrp, lane, acc, accx);
#pragma unroll
            for (int nt = 0; nt < 5; ++nt) tile_store_bias<RP, true>(h2T, b1, 16 * wrp + mg, 8 * nt + mt2, acc[nt], true);
            if (wrp < 5) tile_store_bias<RP, true>(h2T, b1, 192 + mg, 8 * wrp + mt2, accx, false);
        }
        MAIN_SYNC();
        TL3(3);
        {
            const int wrp = tid >> 5, mg = lane >> 2, mt2 = 2 * (lane & 3);
            float acc[3][4], accx[4];
            rowgemm_mma<RP, H, L, 3>(h2T, W2T, wrp, lane, acc, accx);
#pragma unroll
            for (int nt = 0; nt < 3; ++nt)
                if (8 * nt + mt2 < L) tile_store_bias<RP, false>(fT, b2, 16 * wrp + mg, 8 * nt + mt2, acc[nt], true);   // columns 20..23: padding
            if (wrp < 3 && 8 * wrp + mt2 < L) tile_store_bias<RP, false>(fT, b2, 192 + mg, 8 * wrp + mt2, accx, false);
        }
        MAIN_SYNC();
        TL3(4);
#else
        if (tid < 5 * NQ2) {
            u64 a2[4][4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const u64 bv = *reinterpret_cast<const u64*>(b0 + 8 * cg_rg + 2 * i);
#pragma unroll
                for (int r = 0; r < 4; ++r) a2[r][i] = bv;
            }
            rowgemm4<RP, F, H, 8>(xT, W0T, q_rg, 8 * cg_rg, a2);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                float v[4][2];
#pragma unroll
                for (int r = 0; r < 4; ++r) unpack2(a2[r][i], v[r][0], v[r][1]);
#pragma unroll
                for (int e = 0; e < 2; ++e)
                    *reinterpret_cast<float4*>(h1T + (8 * cg_rg + 2 * i + e) * RP + 4 * q_rg) =
                        make_float4(relu_nan(v[0][e]), relu_nan(v[1][e]), relu_nan(v[2][e]), relu_nan(v[3][e]));
            }
        }
        MAIN_SYNC();
        TL3(2);
        if (tid < 5 * NQ2) {
            u64 a2[4][4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const u64 bv = *reinterpret_cast<const u64*>(b1 + 8 * cg_rg + 2 * i);
#pragma unroll
                for (int r = 0; r < 4; ++r) a2[r][i] = bv;
            }
            rowgemm4<RP, H, H, 8>(h1T, W1T, q_rg, 8 * cg_rg, a2);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                float v[4][2];
#pragma unroll
                for (int r = 0; r < 4; ++r) unpack2(a2[r][i], v[r][0], v[r][1]);
#pragma unroll
                for (int e = 0; e < 2; ++e)
                    *reinterpret_cast<float4*>(h2T + (8 * cg_rg + 2 * i + e) * RP + 4 * q_rg) =
                        make_float4(relu_nan(v[0][e]), relu_nan(v[1][e]), relu_nan(v[2][e]), relu_nan(v[3][e]));
            }
        }
        MAIN_SYNC();
        TL3(3);
        if (tid < 5 * NQ2) {
            u64 a2[4][2];
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const u64 bv = *reinterpret_cast<const u64*>(b2 + 4 * cg_rg + 2 * i);
#pragma unroll
                for (int r = 0; r < 4; ++r) a2[r][i] = bv;
            }
            rowgemm4<RP, H, L, 4>(h2T, W2T, q_rg, 4 * cg_rg, a2);
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                float v[4][2];
#pragma unroll
                for (int r = 0; r < 4; ++r) unpack2(a2[r][i], v[r][0], v[r][1]);
#pragma unroll
                for (int e = 0; e < 2; ++e)
                    *reinterpret_cast<float4*>(fT + (4 * cg_rg + 2 * i + e) * RP + 4 * q_rg) =
                        make_float4(v[0][e], v[1][e], v[2][e], v[3][e]);
            }
        }
        MAIN_SYNC();
        TL3(4);
#endif
        // ---- S4: pooling per system (two-pass mean / unbiased variance per latent column, :418-419) ----
        if (lt < L * 8) {
            const int c = lt >> 3, part = lt & 7;
            const float* fc = fT + c * RP + half * T;
            // the column's 25 row quads: this lane takes quads part, part + 8, part + 16 (and 24 when part == 0)
            float4 v[4];
#pragma unroll
            for (int i = 0; i < 4; ++i)
                v[i] = (part + 8 * i < NQ) ? *reinterpret_cast<const float4*>(fc + 4 * (part + 8 * i)) : make_float4(0.f, 0.f, 0.f, 0.f);
            float s = 0.f;
#pragma unroll
            for (int i = 0; i < 4; ++i) s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
            s += __shfl_xor_sync(0xffffffffu, s, 1);
            s += __shfl_xor_sync(0xffffffffu, s, 2);
            s += __shfl_xor_sync(0xffffffffu, s, 4);
            const float mean = __fdiv_rn(s, Tf);
            float m2 = 0.f;
#pragma unroll
            for (int i = 0; i < 4; ++i)
                if (part + 8 * i < NQ) {
                    const float d0 = v[i].x - mean, d1 = v[i].y - mean, d2 = v[i].z - mean, d3 = v[i].w - mean;
                    m2 = fmaf(d0, d0, m2); m2 = fmaf(d1, d1, m2); m2 = fmaf(d2, d2, m2); m2 = fmaf(d3, d3, m2);
                }
            m2 += __shfl_xor_sync(0xffffffffu, m2, 1);
            m2 += __shfl_xor_sync(0xffffffffu, m2, 2);
            m2 += __shfl_xor_sync(0xffffffffu, m2, 4);
            if (part == 0) {
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
                if (act) a_skl += 0.5f * (mus * mus + cst[C3_KLC + c]) + 0.5f * (sds * sds + cst[C3_KLC + L + c]);
            }
        }
        MAIN_SYNC();
        TL3(11);
        // ---- S6: regress_nn forward ----
        if (lt < H * 4) {
            const int j = lt >> 2, part = lt & 3;
            const float* w = V0s + j * S2 + 10 * part;
            float a = 0.f;
#pragma unroll
            for (int k = 0; k < 10; ++k) a = fmaf(sv[V3_SP + 10 * part + k], w[k], a);
            a += __shfl_xor_sync(0xffffffffu, a, 1);
            a += __shfl_xor_sync(0xffffffffu, a, 2);
            if (part == 0) sv[V3_R1 + j] = relu_nan(a + cbs[j]);
        }
        MAIN_SYNC();
        TL3(12);
        if (lt < H * 4) {
            const int j = lt >> 2, part = lt & 3;
            const float* w = V1s + j * H + 10 * part;
            float a = 0.f;
#pragma unroll
            for (int k = 0; k < 10; ++k) a = fmaf(sv[V3_R1 + 10 * part + k], w[k], a);
            a += __shfl_xor_sync(0xffffffffu, a, 1);
            a += __shfl_xor_sync(0xffffffffu, a, 2);
            if (part == 0) sv[V3_R2 + j] = relu_nan(a + cbs[H + j]);
        }
        MAIN_SYNC();
        TL3(13);
        float gr0 = 0.f, gr1 = 0.f;   // valid in the first warp of each half
        if (lt < 32) {
            const int o = lane >> 4, l16 = lane & 15;
            float a = 0.f;
            for (int k = l16; k < H; k += 16) a = fmaf(sv[V3_R2 + k], V2s[o * H + k], a);
            a += __shfl_xor_sync(0xffffffffu, a, 1);
            a += __shfl_xor_sync(0xffffffffu, a, 2);
            a += __shfl_xor_sync(0xffffffffu, a, 4);
            a += __shfl_xor_sync(0xffffffffu, a, 8);
            const float r0 = __shfl_sync(0xffffffffu, a, 0) + cbs[2 * H];
            const float r1 = __shfl_sync(0xffffffffu, a, 16) + cbs[2 * H + 1];
            {
                // lanes 0 and 1 each take one label's truncated-normal term (the longest single-lane chain of the head)
                const float t0 = tanhf(r0), t1 = tanhf(r1);
                const float mu = __fadd_rn(__fmul_rn(__fmul_rn(0.5f, __fadd_rn(t0, 1.0f)), __fsub_rn(prm.hc.hi_mu, prm.hc.lo_mu)), prm.hc.lo_mu);
                const float sd = __fadd_rn(__fmul_rn(__fmul_rn(0.5f, __fadd_rn(t1, 1.0f)), __fsub_rn(prm.hc.hi_sd, prm.hc.lo_sd)), prm.hc.lo_sd);
                float l = 0.f, dm = 0.f, ds = 0.f;
                if (prm.saliency) {   // upstream gradient of mu.sum(): d mu = 1, d sd = 0 (feature_importance.py:109-110)
                    dm = lane == 0 ? -1.0f : 0.f;
                    if (lane == 0 && act) prm.mu_out[sb] = mu;
                } else if (lane < 2) nll_terms(mu, sd, sv[V3_Y + lane], l, dm, ds);
                const float l1 = __shfl_sync(0xffffffffu, l, 1), dm1 = __shfl_sync(0xffffffffu, dm, 1), ds1 = __shfl_sync(0xffffffffu, ds, 1);
                if (lane == 0) {
                    if (act) a_nll += -(l + l1);
                    const float gmu = -(dm + dm1), gsd = -(ds + ds1);
                    // an inactive slot (odd batch tail) contributes nothing: zero upstream gradient
                    gr0 = act ? gmu * 0.5f * (prm.hc.hi_mu - prm.hc.lo_mu) * (1.0f - t0 * t0) : 0.f;
                    gr1 = act ? gsd * 0.5f * (prm.hc.hi_sd - prm.hc.lo_sd) * (1.0f - t1 * t1) : 0.f;
                }
            }
            // ---- S7: regress_nn backward (the same warp carries on: g_a2 = (V2^T g_r) . [r2 > 0]) ----
            gr0 = __shfl_sync(0xffffffffu, gr0, 0);
            gr1 = __shfl_sync(0xffffffffu, gr1, 0);
            for (int k = lane; k < H; k += 32) {
                const float g = gr0 * V2s[k] + gr1 * V2s[H + k];
                sv[V3_G2 + k] = sv[V3_R2 + k] > 0.f ? g : 0.f;
            }
        }
        MAIN_SYNC();
        TL3(14);
        if (lt < H * 4) {
            const int k = lt >> 2, part = lt & 3;
            float a = 0.f;
#pragma unroll
            for (int jj = 0; jj < 10; ++jj) {
                const int j = 10 * part + jj;
                a = fmaf(sv[V3_G2 + j], V1s[j * H + k], a);
            }
            a += __shfl_xor_sync(0xffffffffu, a, 1);
            a += __shfl_xor_sync(0xffffffffu, a, 2);
            if (part == 0) sv[V3_G1 + k] = sv[V3_R1 + k] > 0.f ? a : 0.f;
        }
        MAIN_SYNC();
        TL3(15);
        float* rec = prm.head_rec + sb * REC;
        if (lt < S2 * 4) {
            const int k = lt >> 2, part = lt & 3;
            float a = 0.f;
#pragma unroll
            for (int jj = 0; jj < 10; ++jj) {
                const int j = 10 * part + jj;
                a = fmaf(sv[V3_G1 + j], V0s[j * S2 + k], a);
            }
            a += __shfl_xor_sync(0xffffffffu, a, 1);
            a += __shfl_xor_sync(0xffffffffu, a, 2);
            if (part == 0) {
                if (act && !prm.saliency) rec[R_DLVS + k] = a * (0.5f * (sv[V3_ESN + k] * cst[C3_ELVH + k]));  // ds'/dlv = eps e^{lv/2} / 2
                sv[V3_GS + k] = a + (act ? prm.beta_out[prm.saliency ? 0 : blockIdx.y] * sv[V3_S + k] : 0.f);
            }
        } else if (act && !prm.saliency) {
            // the other warp of the half writes the record (s', r1, r2, g_a1, g_a2 are complete)
            const int i0 = lt - S2 * 4;  // 0..31
            for (int i = i0; i < R_DLVS; i += HALF3 - S2 * 4) rec[i] = sv[V3_REC0 + i];
        }
        if (lt == 0 && act && !prm.saliency) { rec[R_GR] = gr0; rec[R_GR + 1] = gr1; }
        MAIN_SYNC();
        TL3(16);
        // ---- S8: g_f in place over f (each half its own system): g_f[t] = g_m / n + g_v 2 (f_t - m) / (n - 1), the two
        // coefficients recomputed per item from the pooled statistics (cheaper than a 20-thread phase and its barrier) ----
        for (int i = lt; i < L * NQ; i += HALF3) {
            const int c = i / NQ, q = i - c * NQ;
            const float gmus = sv[V3_GS + c], gsds = sv[V3_GS + L + c];
            const float vs = sv[V3_VS + c], sds = sv[V3_S + L + c], var = sv[V3_VAR + c];
            const float sgn = vs > 0.f ? 1.0f : (vs < 0.f ? -1.0f : 0.f);
            const float gvs = gsds * sgn / (2.0f * sds);
            const float e1 = sv[V3_E12 + c], e2 = sv[V3_E12 + L + c];
            const float gv = gmus * e1 / (2.0f * Tf * sv[V3_SIM + c]) +
                             gvs * (1.0f + e2 * (2.0f * var) / (Tm1 * sv[V3_SIV + c]));
            const float A = act ? gmus / Tf : 0.f;        // coefficient of 1
            const float Bc = act ? 2.0f * gv / Tm1 : 0.f;  // coefficient of (f - m)
            float4* p = reinterpret_cast<float4*>(fT + c * RP + half * T + 4 * q);
            const float m = sv[V3_M + c];
            float4 f = *p;
            f.x = fmaf(Bc, f.x - m, A); f.y = fmaf(Bc, f.y - m, A); f.z = fmaf(Bc, f.z - m, A); f.w = fmaf(Bc, f.w - m, A);
            *p = f;
        }
        MAIN_SYNC();
        TL3(5);
        if (tid >= 256 && tid < 256 + L) {  // b2 gradient: fixed-order column sums of g_f (a warp without a GEMM tile)
            const float* g = fT + (tid - 256) * RP;
            float s = 0.f;
            for (int r = 0; r < RT; r += 4) {
                const float4 v = *reinterpret_cast<const float4*>(g + r);
                s += (v.x + v.y) + (v.z + v.w);
            }
            ab2 += s;
        }
        // ---- S10: g_a2 = (g_f W2) . [h2 > 0] ----
#if V3_GEMM == 1
        {
            const int wrp = tid >> 5, mg = lane >> 2, mt2 = 2 * (lane & 3);
            float acc[5][4], accx[4];
            rowgemm_mma<RP, L, H, 5>(fT, W2n, wrp, lane, acc, accx);
#pragma unroll
            for (int nt = 0; nt < 5; ++nt) tile_store_masked<RP>(g2T, h2T, 16 * wrp + mg, 8 * nt + mt2, acc[nt], true);
            if (wrp < 5) tile_store_masked<RP>(g2T, h2T, 192 + mg, 8 * wrp + mt2, accx, false);
        }
        MAIN_SYNC();
        TL3(6);
#else
        if (tid < 5 * NQ2) {
            u64 a2[4][4];
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int i = 0; i < 4; ++i) a2[r][i] = 0ull;
            rowgemm4<RP, L, H, 8>(fT, W2n, q_rg, 8 * cg_rg, a2);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                float v[4][2];
#pragma unroll
                for (int r = 0; r < 4; ++r) unpack2(a2[r][i], v[r][0], v[r][1]);
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int col = 8 * cg_rg + 2 * i + e;
                    const float4 h = *reinterpret_cast<const float4*>(h2T + col * RP + 4 * q_rg);
                    *reinterpret_cast<float4*>(g2T + col * RP + 4 * q_rg) =
                        make_float4(h.x > 0.f ? v[0][e] : 0.f, h.y > 0.f ? v[1][e] : 0.f, h.z > 0.f ? v[2][e] : 0.f,
                                    h.w > 0.f ? v[3][e] : 0.f);
                }
            }
        }
        MAIN_SYNC();
        TL3(6);
#endif
        // ---- S12: g_a1 = (g_a2 W1) . [h1 > 0] ----
#if V3_GEMM == 1
        {
            const int wrp = tid >> 5, mg = lane >> 2, mt2 = 2 * (lane & 3);
            float acc[5][4], accx[4];
            rowgemm_mma<RP, H, H, 5>(g2T, W1n, wrp, lane, acc, accx);
#pragma unroll
            for (int nt = 0; nt < 5; ++nt) tile_store_masked<RP>(g1T, h1T, 16 * wrp + mg, 8 * nt + mt2, acc[nt], true);
            if (wrp < 5) tile_store_masked<RP>(g1T, h1T, 192 + mg, 8 * wrp + mt2, accx, false);
        }
        MAIN_SYNC();
        TL3(7);
#else
        if (tid < 5 * NQ2) {
            u64 a2[4][4];
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int i = 0; i < 4; ++i) a2[r][i] = 0ull;
            rowgemm4<RP, H, H, 8>(g2T, W1n, q_rg, 8 * cg_rg, a2);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                float v[4][2];
#pragma unroll
                for (int r = 0; r < 4; ++r) unpack2(a2[r][i], v[r][0], v[r][1]);
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int col = 8 * cg_rg + 2 * i + e;
                    const float4 h = *reinterpret_cast<const float4*>(h1T + col * RP + 4 * q_rg);
                    *reinterpret_cast<float4*>(g1T + col * RP + 4 * q_rg) =
                        make_float4(h.x > 0.f ? v[0][e] : 0.f, h.y > 0.f ? v[1][e] : 0.f, h.z > 0.f ? v[2][e] : 0.f,
                                    h.w > 0.f ? v[3][e] : 0.f);
                }
            }
        }
        MAIN_SYNC();
        TL3(7);
#endif
        // ---- S13: all weight-gradient outer products in one phase ----
        if (!prm.saliency) {
#if V3_OUTER == 16
            {   // column tiles 0..2, then 3..4 (dW2 has three): at most 36 accumulators in registers at a time
                float a3[3][16];
                stash_load<48>(taddr, &a3[0][0]);
                outer_mma<RP, 3>(opH, opG, op_q0, op_q1, lane, a3);
                stash_store<48>(taddr, &a3[0][0]);
            }
            if (op_role < 2) {
                float a2[2][16];
                stash_load<32>(taddr + 48, &a2[0][0]);
                outer_mma<RP, 2>(opH, opG + 24 * RP, op_q0, op_q1, lane, a2);
                stash_store<32>(taddr + 48, &a2[0][0]);
            }
#else
            float aW[OJ][8];
            stash_load<NV>(taddr, &aW[0][0]);
#if V3_OUTER == 88
            outer8x8(opG, op_gstr, opH, 5 * RP, op_q0, op_q1, aW);
#else
            outer4x8(opG, op_gstr, opH, 5 * RP, op_q0, op_q1, aW);
#endif
            stash_store<NV>(taddr, &aW[0][0]);
#endif
        }
        TL3(8);
        // ---- S14: g_x = g_a1 W0, dlv_in += sum g_x . (x' - mask(x)) / 2; the two spare warps do the row sums ----
#if V3_GEMM == 1
        {
            const int wrp = tid >> 5, mg = lane >> 2, mt2 = 2 * (lane & 3);
            // n = x' - mask(x) of this thread's elements, from the L2 scratch: issued before the GEMM so that the latency
            // hides under it (slot nt: columns 8 nt + 2 t + e, rows 16 w + g (+8); slot 6: the 13th row tile)
            float nn[7][4];
            if (!prm.saliency) {
#pragma unroll
                for (int nt = 0; nt < 7; ++nt) {
                    const int row = nt < 6 ? 16 * wrp + mg : 192 + mg, col = nt < 6 ? 8 * nt + mt2 : 8 * wrp + mt2;
                    const bool full = nt < 6;
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const int cc = min(col + e, F - 1);
                        nn[nt][e] = (nt < 6 || wrp < 6) ? __ldcg(np_cur + cc * RT + row) : 0.f;
                        nn[nt][2 + e] = full ? __ldcg(np_cur + cc * RT + row + 8) : 0.f;
                    }
                }
            }
            float acc[6][4], accx[4];
            rowgemm_mma<RP, H, W0NP, 6>(g1T, W0n, wrp, lane, acc, accx);
            float agx[8][2];
            stash_load<16>(taddr + NV, &agx[0][0]);
            // one tile: d mu / d x (saliency) or dlv_in += g_x . (x' - mask(x)), with n = x' - mask(x) from the L2 scratch
            auto tile = [&](int row, int col, const float (&c)[4], bool full, float (&ag)[2], const float (&nv)[4]) {
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int cc = col + e;
                    if (cc < F) {
                        const float v0 = c[e], v1 = full ? c[2 + e] : 0.f;
                        if (prm.saliency) {
                            ag[e] += fmaf(v0, v0, v1 * v1);
                            if (prm.gx_out) {
#pragma unroll
                                for (int h8 = 0; h8 < 2; ++h8) {
                                    const int rr = row + 8 * h8, hs = rr >= T ? 1 : 0, bb = b0i + hs;
                                    if ((h8 == 0 || full) && bb < prm.B)
                                        prm.gx_out[(((int64_t)sidx * prm.B + bb) * T + rr - hs * T) * F + cc] = h8 ? v1 : v0;
                                }
                            }
                        } else {
                            ag[e] += fmaf(v0, nv[e], v1 * nv[2 + e]);
                        }
                    }
                }
            };
#pragma unroll
            for (int nt = 0; nt < 6; ++nt) tile(16 * wrp + mg, 8 * nt + mt2, acc[nt], true, agx[nt], nn[nt]);
            if (wrp < 6) tile(192 + mg, 8 * wrp + mt2, accx, false, agx[6], nn[6]);
            stash_store<16>(taddr + NV, &agx[0][0]);
            if (!prm.saliency && tid < 2 * H) {   // b0 = row sums of g_a1, b1 = row sums of g_a2
                const float* gsrc = tid < H ? g1T + tid * RP : g2T + (tid - H) * RP;
                float s0 = 0.f, s1 = 0.f;
                for (int tt = 0; tt < RT; tt += 4) {
                    const float4 v = *reinterpret_cast<const float4*>(gsrc + tt);
                    s0 += v.x + v.z; s1 += v.y + v.w;
                }
                arow += s0 + s1;
            }
        }
#else
        if (tid < 6 * NQ2) {
            u64 a2[4][4];
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int i = 0; i < 4; ++i) a2[r][i] = 0ull;
            // n = x' - mask(x) of these rows comes back from the scratch (inactive slots hold zeros); the L2 loads are
            // issued before the GEMM so that their latency hides under it
            float4 nn[8];
#pragma unroll
            for (int c = 0; c < 8; ++c)
                nn[c] = __ldcg(reinterpret_cast<const float4*>(np_cur + min(8 * cg_rg + c, F - 1) * RT) + q_rg);
            rowgemm4<RP, H, W0NP, 8>(g1T, W0n, q_rg, 8 * cg_rg, a2);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                float v[4][2];
#pragma unroll
                for (int r = 0; r < 4; ++r) unpack2(a2[r][i], v[r][0], v[r][1]);
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int col = 8 * cg_rg + 2 * i + e;
                    if (col < F) {
                        if (prm.saliency) {   // d mu / d x: sum of squares per column, and the rows themselves if asked for
                            aux[2 * i + e] += fmaf(v[0][e], v[0][e], fmaf(v[1][e], v[1][e], fmaf(v[2][e], v[2][e], v[3][e] * v[3][e])));
                            const int hs = q_rg / NQ, bb = b0i + hs;
                            if (prm.gx_out && bb < prm.B) {
                                float* o = prm.gx_out + (((int64_t)sidx * prm.B + bb) * T + 4 * (q_rg - hs * NQ)) * F + col;
#pragma unroll
                                for (int r = 0; r < 4; ++r) o[r * F] = v[r][e];
                            }
                        } else {
                            const float4 n4 = nn[2 * i + e];
                            aux[2 * i + e] += fmaf(v[0][e], n4.x, fmaf(v[1][e], n4.y, fmaf(v[2][e], n4.z, v[3][e] * n4.w)));
                        }
                    }
                }
            }
        } else if (!prm.saliency) {
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int r = tid - 6 * NQ2 + e * (NMAIN - 6 * NQ2);  // 84 threads, rows r and r + 84 of 120
#if V3_OUTER == 16
                if (r < 3 * H && (r < H || r >= 2 * H)) {   // column 40 of dW0 is covered by the tensor-core tiles
#else
                if (r < 3 * H) {
#endif
                    const float* g = r < 2 * H ? g1T + (r < H ? r : r - H) * RP : g2T + (r - 2 * H) * RP;
                    float s0 = 0.f, s1 = 0.f;
                    if (r >= H && r < 2 * H) {
                        const float* xc = xT + (F - 1) * RP;
                        for (int t = 0; t < RT; t += 4) {
                            const float4 v = *reinterpret_cast<const float4*>(g + t);
                            const float4 x = *reinterpret_cast<const float4*>(xc + t);
                            s0 = fmaf(v.x, x.x, s0); s1 = fmaf(v.y, x.y, s1); s0 = fmaf(v.z, x.z, s0); s1 = fmaf(v.w, x.w, s1);
                        }
                    } else {
                        for (int t = 0; t < RT; t += 4) {
                            const float4 v = *reinterpret_cast<const float4*>(g + t);
                            s0 += v.x + v.z; s1 += v.y + v.w;
                        }
                    }
                    aux[e] += s0 + s1;
                }
            }
        }
#endif
        if (b0i + 4 * (int)gridDim.x < prm.B) nb_arrive(3 + parity, NTHR3);   // this parity's scratch may be overwritten
        MAIN_SYNC();
        TL3(9);
        parity ^= 1;
    }

    // =====================================================================================================
    // Epilogue: this CTA's partial gradient in flatten() order.  The activation buffers are dead: scratch.
    // =====================================================================================================
    float* part = prm.partial + ((int64_t)sidx * prm.n_cta + blockIdx.x) * (fl.d + DPAD);
    float* red = sm;  // up to 45,084 floats
    // (1) feature matrices: add the row groups in a fixed order
    float aW[OJ][8];
    stash_load<NV>(taddr, &aW[0][0]);
#if V3_OUTER == 16
    {
        // every warp parks its 60 partial sums; the first warp of a matrix adds its partners' in warp order and writes
        float* o = red + tid * 80;
#pragma unroll
        for (int i = 0; i < 80; ++i) o[i] = (&aW[0][0])[i];
        MAIN_SYNC();
        const int first = op_role == 0 ? 0 : (op_role == 1 ? 5 : 10), nw = op_role == 2 ? 2 : 5;
        if (owarp == first) {
            const int nnt = op_role == 2 ? 3 : 5;
            const int g = lane >> 2, t = lane & 3;
            const int off = op_role == 0 ? fl.W0 : (op_role == 1 ? fl.W1 : fl.W2);
            const int pitch = op_role == 0 ? F : H, mmax = op_role == 0 ? F : H, nmax = op_role == 2 ? L : H;
            for (int mt = 0; mt < 3; ++mt)
                for (int nt = 0; nt < nnt; ++nt)
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const int idx = nt * 16 + mt * 4 + i;
                        float a = 0.f;
                        for (int w = 0; w < nw; ++w) a += red[((first + w) * 32 + lane) * 80 + idx];
                        const int m = 16 * mt + g + (i & 2 ? 8 : 0), n = 8 * nt + 2 * t + (i & 1);
                        if (m < mmax && n < nmax) part[off + n * pitch + m] = a;
                    }
        }
    }
#else
    if (op_role < 3) {
        float* o = red + tid * (OJ * 8);
#pragma unroll
        for (int jj = 0; jj < OJ; ++jj)
#pragma unroll
            for (int kk = 0; kk < 8; ++kk) o[jj * 8 + kk] = aW[jj][kk];
    }
#endif
    MAIN_SYNC();
#if V3_OUTER != 16
    if (op_role < 3) {
#if V3_OUTER == 88
        const int nblk = op_role == 2 ? 15 : 25, ngrp = op_role == 2 ? 5 : 6;
        const int jstr = op_role == 2 ? 3 : 5;
#else
        const int nblk = op_role == 2 ? 25 : 50, ngrp = 3;
        const int jstr = op_role == 2 ? 5 : 10;
#endif
        const int jmax = op_role == 2 ? L : H;
        const int base = op_role == 0 ? 0 : (op_role == 1 ? 150 : 300);
        if (tid - base < nblk) {  // the row-group-0 owner of the block sums and writes
            const int off = op_role == 0 ? fl.W0 : (op_role == 1 ? fl.W1 : fl.W2);
            const int pitch = op_role == 0 ? F : H;
#pragma unroll
            for (int jj = 0; jj < OJ; ++jj)
#pragma unroll
                for (int kk = 0; kk < 8; ++kk) {
                    float a = aW[jj][kk];
                    for (int g = 1; g < ngrp; ++g) a += red[(tid + g * nblk) * (OJ * 8) + jj * 8 + kk];
                    const int j = op_jb + jstr * jj;
                    if (j < jmax) part[off + j * pitch + op_kb + 5 * kk] = a;
                }
        }
    }
#endif
    MAIN_SYNC();
    // (2) dlv_in (fixed-order sum over the row quads), b0 / b1 / column 40 of dW0, b2
#if V3_GEMM == 1
    {
        // thread (warp w, g, t) holds, for column tile nt (slot nt) and e: the sum over its rows of column 8 nt + 2 t + e;
        // slot 6 (warps 0..5): the 13th row tile, column 8 w + 2 t + e.  red[col][w * 8 + g] / red[col][96 + g].
        const int wrp = tid >> 5, g = lane >> 2, t = lane & 3;
        float agx[8][2];
        stash_load<16>(taddr + NV, &agx[0][0]);
#pragma unroll
        for (int nt = 0; nt < 6; ++nt)
#pragma unroll
            for (int e = 0; e < 2; ++e) red[(8 * nt + 2 * t + e) * 104 + wrp * 8 + g] = agx[nt][e];
        if (wrp < 6) {
#pragma unroll
            for (int e = 0; e < 2; ++e) red[(8 * wrp + 2 * t + e) * 104 + 96 + g] = agx[6][e];
        }
        if (tid < H) part[fl.b0 + tid] = arow;
        else if (tid < 2 * H) part[fl.b1 + tid - H] = arow;
        if (tid >= 256 && tid < 256 + L) part[fl.b2 + tid - 256] = ab2;
        MAIN_SYNC();
        if (tid < F) {
            float sacc = 0.f;
            for (int i = 0; i < 104; ++i) sacc += red[tid * 104 + i];
            part[fl.lv_in + tid] = 0.5f * sacc;
        }
        MAIN_SYNC();
    }
#else
    if (tid < 6 * NQ2) {
#pragma unroll
        for (int c = 0; c < 8; ++c) red[(8 * cg_rg + c) * NQ2 + q_rg] = aux[c];
    } else {
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int r = tid - 6 * NQ2 + e * (NMAIN - 6 * NQ2);
            if (r < H) part[fl.b0 + r] = aux[e];
            else if (r < 2 * H) {
#if V3_OUTER != 16
                part[fl.W0 + (r - H) * F + (F - 1)] = aux[e];   // (the tensor-core tiles cover column 40 themselves)
#endif
            }
            else if (r < 3 * H) part[fl.b1 + r - 2 * H] = aux[e];
        }
    }
    if (tid >= 256 && tid < 256 + L) part[fl.b2 + tid - 256] = ab2;
    MAIN_SYNC();
    if (tid < F) {
        float s = 0.f;
        for (int q = 0; q < NQ2; ++q) s += red[tid * NQ2 + q];
        part[fl.lv_in + tid] = 0.5f * s;
    }
    MAIN_SYNC();
#endif
    // (3) metrics: nll (lane 0 of the first warp of each half) and the summary KL (pooling threads with part == 0)
    red[tid] = (lt < L * 8 && (lt & 7) == 0) ? a_skl : 0.f;
    red[NMAIN + tid] = (lt == 0) ? a_nll : 0.f;
    MAIN_SYNC();
    if (tid == 0) {
        float s = 0.f;
        for (int h = 0; h < 2; ++h)
            for (int c = 0; c < L; ++c) s += red[h * HALF3 + 8 * c];
        part[fl.d + SLOT_NLL] = red[NMAIN] + red[NMAIN + HALF3];
        part[fl.d + SLOT_SKL] = s;
        for (int i = 2; i < DPAD; ++i) part[fl.d + i] = 0.f;
    }
    MAIN_SYNC();
    // (4) head gradients from the records of this CTA's systems, in system order:
    //     dV0 += g_a1 s'^T, c0 += g_a1; dV1 += g_a2 r1^T, c1 += g_a2; dV2 += g_r r2^T, c2 += g_r; dlv_sum += dlvs
    if (!prm.saliency) {
        constexpr int CH = 128;  // records staged per chunk (128 kB)
        // roles: tid < 200: 2 x 4 blocks of dV0 and dV1; 200..239: c0, c1; 240..319: dV2; 320..321: c2; 322..361: dlv_sum
        const int jbh = tid / 10, kb = tid % 10;
        float aV0[2][4] = {}, aV1[2][4] = {};
        float s0 = 0.f, s1 = 0.f;
        const int n_it = (prm.B - 2 * (int)blockIdx.x + 2 * (int)gridDim.x - 1) / (2 * (int)gridDim.x);  // loop trips
        const int n_sys = 2 * n_it;  // slots (the last one may be past the batch)
        for (int c0i = 0; c0i < n_sys; c0i += CH) {
            const int nc = min(CH, n_sys - c0i);
            for (int i = tid; i < nc * (REC / 4); i += NMAIN) {
                const int s = c0i + i / (REC / 4), w = i % (REC / 4);
                const int bsys = 2 * blockIdx.x + 2 * gridDim.x * (s >> 1) + (s & 1);
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (bsys < prm.B)
                    v = __ldcg(reinterpret_cast<const float4*>(prm.head_rec + ((int64_t)sidx * prm.B + bsys) * REC) + w);
                reinterpret_cast<float4*>(red)[i] = v;
            }
            MAIN_SYNC();
            if (tid < 200) {
                for (int s = 0; s < nc; ++s) {
                    const float* r = red + s * REC;
#pragma unroll
                    for (int jj = 0; jj < 2; ++jj)
#pragma unroll
                        for (int kk = 0; kk < 4; ++kk) {
                            aV0[jj][kk] = fmaf(r[R_G1 + 2 * jbh + jj], r[R_SP + kb + 10 * kk], aV0[jj][kk]);
                            aV1[jj][kk] = fmaf(r[R_G2 + 2 * jbh + jj], r[R_R1 + kb + 10 * kk], aV1[jj][kk]);
                        }
                }
            } else if (tid < 240) {
                for (int s = 0; s < nc; ++s) { s0 += red[s * REC + R_G1 + tid - 200]; s1 += red[s * REC + R_G2 + tid - 200]; }
            } else if (tid < 320) {
                const int o = (tid - 240) / H, k = (tid - 240) % H;
                for (int s = 0; s < nc; ++s) s0 = fmaf(red[s * REC + R_GR + o], red[s * REC + R_R2 + k], s0);
            } else if (tid < 322) {
                for (int s = 0; s < nc; ++s) s0 += red[s * REC + R_GR + tid - 320];
            } else if (tid < 322 + S2) {
                for (int s = 0; s < nc; ++s) s0 += red[s * REC + R_DLVS + tid - 322];
            }
            MAIN_SYNC();
        }
        if (tid < 200) {
#pragma unroll
            for (int jj = 0; jj < 2; ++jj)
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {
                    part[fl.V0 + (2 * jbh + jj) * S2 + kb + 10 * kk] = aV0[jj][kk];
                    part[fl.V1 + (2 * jbh + jj) * H + kb + 10 * kk] = aV1[jj][kk];
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
    MAIN_SYNC();
    if (tid < 32) tmem_dealloc(tbase, TCOLS);
    TL3(10);
#ifdef BNN_TRAIN_TIMELINE
    if (tid == 0 && blockIdx.x == 0 && blockIdx.y == 0)
        for (int i = 0; i < 18; ++i) g_train_tl[i] = tl[i];

#endif
}

}  // namespace train
}  // namespace bnn

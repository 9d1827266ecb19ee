// K1 (round 2): batched 32x32 Householder QR, "one lane = one column" form.
//
// Reference semantics: linalg/qr.py:52-100 (householder_qr) for every A[b] of a (batch, 32, 32) array.
//
// Measured facts behind this form (profiles/r2_hh32_notes.md, tools/ubench/dfma_regs.cu, dmma_issue.cu):
//   * a DFMA with three distinct register operands issues every 3 cycles, not 2 (24.4 vs 36.7 TFLOP/s): the batched
//     kernels are bound by operand delivery / issue slots, so every shuffle, select and address instruction of the
//     2-D (row-parity x column-slot) layouts of round 1 costs real time;
//   * a DMMA.8x8x4 (256 FMAs) costs ~6 issue cycles and 16 pipe cycles.
//
//   R phase  four matrices per warp, 8 lanes each, LEFT-LOOKING over four panels of 8 columns: lane c of a group owns
//            column 8p + c with all 32 rows in registers (64 registers).  A panel is loaded, the reflectors of the
//            earlier panels are applied to it (vector broadcast from shared memory, dot product and update are
//            lane-local: no shuffles, no masks, exactly rows j..31), then its 8 columns are factored (one 64-bit
//            shuffle per column for ||x||^2; the scalar chain is shared by four matrices).
//   storage  reflector j = rows (j & ~1)..31 in natural order, pivot patched to v0 (the row above an odd pivot to 0)
//            after the scalar chain: 544 + 32 doubles per matrix.
//   Q phase  compact-WY on DMMA.8x8x4, one matrix at a time on all 32 lanes: Q^T lives in 16 accumulator tiles
//            (32 doubles / lane).  A DMMA.8x8x4 (the only f64 MMA shape sm_100a has; every mma.sync f64 shape lowers to
//            it) does 256 FMAs for one issue slot (the round-1 kernel's rank-1 DFMA Q phase issued ~1 930 FP64 instructions
//            per matrix).
//            G_p = V_p^T V_p (4 panels of 8 reflectors)                         20 DMMA
//            T_p by the dlarft row recurrence, lane (g, t) = row g of panel t    ~36 DFMA for all four panels at once
//            for p = 3..0:  W^T = Q^T V_p ; W2^T = W^T (-T_p)^T ; Q^T += W2^T V_p^T   28 + 20 + 60 DMMA
//            An accumulator fragment IS a valid A operand when the contraction index is permuted (k = t <-> column
//            2t+i), so W^T and W2^T never leave registers; V is read from shared memory directly in B-fragment order.
//
// Tile / fragment conventions (lane l, g = l >> 2, t = l & 3), mma.m8n8k4.f64:
//   A[g][t], B[t][g], C[g][2t], C[g][2t+1].
//   qt[cb][rb][i] = Q[8 rb + 2t + i][8 cb + g]          (tile (cb, rb) of Q^T)
//   F1(p, rb, i)  = V[8 rb + 2t + i][8 p + g]           (B operand of W^T = Q^T V, A and B operand of the Gram)
//   F3(p, rb, i)  = V[8 rb + g][8 p + 2t + i]           (B operand of the update; the panel's own W^T tile)
#pragma once

#include "common.cuh"

namespace lq {

struct Col8 {
    __host__ __device__ static constexpr int r0(int j) { return j & ~1; }
    __host__ __device__ static constexpr int vsize(int j) { return 32 - (j & ~1); }
    __host__ __device__ static constexpr int voff(int j) {  // sum of vsize(t), t < j
        return 2 * (32 * (j >> 1) - (j >> 1) * ((j >> 1) - 1)) + (j & 1) * (32 - 2 * (j >> 1));
    }
    __host__ __device__ static constexpr int voff_slow(int j) {
        int o = 0;
        for (int t = 0; t < j; ++t) o += vsize(t);
        return o;
    }
    static constexpr int VDOUBLES = 544;
    static constexpr int BETA = VDOUBLES;
    static constexpr int MAT = 580;      // 290 16-byte words = 2 (mod 8): the four matrices of a warp hit four different bank quads
    static constexpr int GSTR = 66;      // stride between the 8 x 8 panel blocks of the scratch (33 words: the four panels
                                         // read by one instruction start in four different bank quads)
    static constexpr int SCRATCH = 3 * 4 * GSTR;  // per warp: G of the next-but-one matrix, -T of the current and the next
    static constexpr int WARP_DOUBLES = 4 * MAT + SCRATCH;
};
static_assert(Col8::voff_slow(32) == Col8::VDOUBLES && Col8::voff(32) == Col8::VDOUBLES, "packed size");
static_assert(Col8::voff(7) == Col8::voff_slow(7) && Col8::voff(18) == Col8::voff_slow(18) && Col8::voff(31) == Col8::voff_slow(31),
              "closed-form offsets");

// grid: ceil(batch / (4 WARPS)) blocks of WARPS warps, WARPS * Col8::WARP_DOUBLES doubles of dynamic shared memory.
// The broadcast reflector is kept in registers between dot product and update instead of being re-read.
template <int WARPS, int MINB>
__global__ void __launch_bounds__(WARPS * 32, MINB)
    hh_qr32_c8_kernel(const double* __restrict__ A, double* __restrict__ Q, double* __restrict__ R, long long batch) {
    constexpr int N = 32;
    extern __shared__ __align__(16) double smem[];

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double* wbase = smem + (size_t)warp * Col8::WARP_DOUBLES;
    const long long mat0 = ((long long)blockIdx.x * WARPS + warp) * 4;

    {
        // ================= R phase (four matrices per warp, 8 lanes each, lane = column) =================
        const int g4 = lane >> 3, c = lane & 7;
        const long long mat = mat0 + g4;
        const bool valid = mat < batch;
        const long long matc = valid ? mat : (batch - 1);
        double* vb = wbase + g4 * Col8::MAT;
        double* betas = vb + Col8::BETA;

#pragma unroll
        for (int p = 0; p < 4; ++p) {
            const int col = 8 * p + c;
            double a[N];
            const double* Ag = A + matc * (N * N) + col;
#pragma unroll
            for (int i = 0; i < N; ++i) a[i] = ld_stream(Ag + i * N);

            // ---- apply the reflectors of the earlier panels: a -= beta_j (v_j . a) v_j, rows j..31, all lane-local
#pragma unroll
            for (int j = 0; j < 8 * p; ++j) {
                const int r0 = Col8::r0(j);
                const double* vj = vb + Col8::voff(j) - r0;  // row i of v_j at vj[i]
                double d[4] = {0.0, 0.0, 0.0, 0.0};
                double vk[N];
#pragma unroll
                for (int i = r0; i < N; i += 2) {
                    const double2 vv = *reinterpret_cast<const double2*>(vj + i);
                    vk[i] = vv.x, vk[i + 1] = vv.y;
                    d[(i >> 1) & 1] = fma(vv.x, a[i], d[(i >> 1) & 1]);
                    d[2 + ((i >> 1) & 1)] = fma(vv.y, a[i + 1], d[2 + ((i >> 1) & 1)]);
                }
                const double s = betas[j] * ((d[0] + d[1]) + (d[2] + d[3]));
#pragma unroll
                for (int i = r0; i < N; ++i) a[i] = fma(-s, vk[i], a[i]);
            }

            // ---- factor the 8 columns of this panel
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) {
                const int j = 8 * p + jj;
                const int r0 = Col8::r0(j);
                const bool odd = (j & 1) != 0;
                double* vj = vb + Col8::voff(j) - r0;

                if (c == jj) {
#pragma unroll
                    for (int i = r0; i < N; i += 2) *reinterpret_cast<double2*>(vj + i) = make_double2(a[i], a[i + 1]);
                }
                __syncwarp();

                // first row pair: the row above an odd pivot belongs to R, not to x
                double2 vf = *reinterpret_cast<const double2*>(vj + r0);
                if (odd) vf.x = 0.0;
                const double x0 = odd ? vf.y : vf.x;

                double d[4];
                double vk[N];
                d[0] = vf.x * a[r0];
                d[2] = vf.y * a[r0 + 1];
                d[1] = 0.0;
                d[3] = 0.0;
#pragma unroll
                for (int i = r0 + 2; i < N; i += 2) {
                    const double2 vv = *reinterpret_cast<const double2*>(vj + i);
                    vk[i] = vv.x, vk[i + 1] = vv.y;
                    d[(i >> 1) & 1] = fma(vv.x, a[i], d[(i >> 1) & 1]);
                    d[2 + ((i >> 1) & 1)] = fma(vv.y, a[i + 1], d[2 + ((i >> 1) & 1)]);
                }
                const double dot = (d[0] + d[1]) + (d[2] + d[3]);            // x^T a_c
                const double ss = __shfl_sync(0xffffffffu, dot, jj, 8);      // ||x||^2 = the owner column's own dot product

                const double ssc = fmax(ss, 1e-300);
                // y = 1/||x||, beta = 2 / v^T v = y^2 / (1 + |x0| y); the reciprocal is seeded from the UNREFINED y
                const double ax0 = fabs(x0);
                double y = rsqrt_seed(ssc);
                double u = rcp_seed(fma(ax0, y, 1.0));
                const double hx = 0.5 * ssc;
#pragma unroll
                for (int it = 0; it < 2; ++it) {
                    const double e = fma(-hx * y, y, 0.5);
                    y = fma(y, e, y);
                }
                const double nrm = ssc * y;
                const double Dn = fma(ax0, y, 1.0);
#pragma unroll
                for (int it = 0; it < 2; ++it) {
                    const double e = fma(-Dn, u, 1.0);
                    u = fma(u, e, u);
                }
                double beta = (y * y) * u;
                const bool skip = nrm < kEps;  // qr.py:79-80
                const double alpha = copysign(nrm, x0);
                const double v0 = x0 + alpha;
                beta = skip ? 0.0 : beta;

                // v^T a_c = x^T a_c + alpha * a[j][c]
                const double s = beta * fma(alpha, a[j], dot);

                // first pair with the pivot element v0, stored back for the later panels and the Q phase
                if (odd) vf.y = v0;
                else vf.x = v0;
                __syncwarp();  // every lane has read the raw first pair
                if (c == jj) *reinterpret_cast<double2*>(vj + r0) = vf;
                if (c == 0) betas[j] = beta;

                a[r0] = fma(-s, vf.x, a[r0]);
                a[r0 + 1] = fma(-s, vf.y, a[r0 + 1]);
#pragma unroll
                for (int i = r0 + 2; i < N; ++i) a[i] = fma(-s, vk[i], a[i]);
                // exact diagonal for the owner (mathematically the update already gives -alpha)
                if (c == jj && !skip) a[j] = -alpha;
            }

            __syncwarp();  // the last pivot patch of this panel is visible to the apply steps of the next one

            // ---- store the R columns of this panel (strict lower triangle forced to exact zeros, qr.py:97)
            if (valid) {
                double* Rg = R + mat * (N * N) + col;
#pragma unroll
                for (int i = 0; i < N; ++i) {
                    double v = a[i];
                    if (i >= 8 * p + 8) v = 0.0;
                    else if (i >= 8 * p) v = (i <= col) ? v : 0.0;
                    st_stream(Rg + i * N, v);
                }
            }
        }
    }
    __syncwarp();

    // ================= Q phase: Q = (I - V0 T0 V0^T) ... (I - V3 T3 V3^T), backward accumulation on DMMA ==========
    // Fragment conventions as in the header comment (g = gq, t = tq).  Software-pipelined over the four
    // matrices of the warp: while the block reflectors of matrix mi are applied (DMMA chains), the T recurrence of matrix
    // mi+1 (a DFMA chain) and the Gram products of matrix mi+2 run in the same instruction stream and fill the bubbles.
    const int gq = lane >> 2, tq = lane & 3;
    double* Gs = wbase + 4 * Col8::MAT;          // 4 panels x GSTR
    double* Ts = Gs + 4 * Col8::GSTR;            // 2 buffers x 4 panels x GSTR (-T of the current / next matrix)
    const bool m1 = gq >= 2 * tq, m1b = gq >= 2 * tq + 1;   // F3 diagonal-tile masks (row g >= column 2t+i)
    const bool m0 = 2 * tq >= gq, m0b = 2 * tq + 1 >= gq;   // F1 diagonal-tile masks (row 2t+i >= column g)
    // V[r][k] lives at voff(k) + r - (k & ~1)
    int f1o[4], f3o[4][2];
#pragma unroll
    for (int p = 0; p < 4; ++p) {
        const int k1 = 8 * p + gq;  // F1: rows 8 rb + 2 tq + {0, 1} (one 16-byte load)
        f1o[p] = Col8::voff(k1) - (k1 & ~1) + 2 * tq;
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const int k3 = 8 * p + 2 * tq + i;  // F3: row 8 rb + gq
            f3o[p][i] = Col8::voff(k3) - (k3 & ~1) + gq;
        }
    }
    auto F1 = [&](const double* vb, int p, int rb) -> double2 {
        double2 v = *reinterpret_cast<const double2*>(vb + f1o[p] + 8 * rb);
        if (rb == p) {
            v.x = m0 ? v.x : 0.0;
            v.y = m0b ? v.y : 0.0;
        }
        return v;
    };
    auto F3 = [&](const double* vb, int p, int rb, int i) -> double {
        double v = vb[f3o[p][i] + 8 * rb];
        if (rb == p) v = (i ? m1b : m1) ? v : 0.0;
        return v;
    };
    // Gram matrices of the four panels of one matrix (accumulator layout)
    auto gram4 = [&](const double* vb, double (&G)[4][2]) {
#pragma unroll
        for (int p = 0; p < 4; ++p) G[p][0] = G[p][1] = 0.0;
        // row block outermost: the four accumulator chains advance together (a lone dependent DMMA chain runs at 55 %)
#pragma unroll
        for (int rb = 3; rb >= 0; --rb) {
            double2 f[4];
#pragma unroll
            for (int p = 0; p <= rb; ++p) f[p] = F1(vb, p, rb);
#pragma unroll
            for (int p = 0; p <= rb; ++p) dmma_8x8x4(G[p], f[p].x, f[p].x);
#pragma unroll
            for (int p = 0; p <= rb; ++p) dmma_8x8x4(G[p], f[p].y, f[p].y);
        }
    };
    auto store_g = [&](const double (&G)[4][2]) {
#pragma unroll
        for (int p = 0; p < 4; ++p) *reinterpret_cast<double2*>(Gs + p * Col8::GSTR + gq * 8 + 2 * tq) = make_double2(G[p][0], G[p][1]);
    };
    // -T of panel tq, row gq (dlarft, forward / columnwise): T[g][k] = -beta_k sum_{m=g}^{k-1} T[g][m] G[m][k]
    auto trec = [&](const double* betas, double (&Tn)[8]) {
        double bk[8], acc[8];
#pragma unroll
        for (int k = 0; k < 8; k += 2) {
            const double2 b2 = *reinterpret_cast<const double2*>(betas + 8 * tq + k);
            bk[k] = b2.x;
            bk[k + 1] = b2.y;
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) acc[k] = 0.0;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            // branch-free: tk = beta_k on the diagonal, -beta_k * acc right of it, 0 left of it
            const double sel = (k == gq) ? 1.0 : 0.0, gt = (k > gq) ? 1.0 : 0.0;
            const double tk = bk[k] * fma(-gt, acc[k], sel);
            Tn[k] = -tk;
            if (k < 7) {
#pragma unroll
                for (int kk = (k + 1) & ~1; kk < 8; kk += 2) {
                    const double2 g2 = *reinterpret_cast<const double2*>(Gs + tq * Col8::GSTR + k * 8 + kk);
                    if (kk > k) acc[kk] = fma(tk, g2.x, acc[kk]);
                    acc[kk + 1] = fma(tk, g2.y, acc[kk + 1]);
                }
            }
        }
    };
    auto store_t = [&](double* Tb, const double (&Tn)[8]) {
#pragma unroll
        for (int k = 0; k < 8; k += 2) *reinterpret_cast<double2*>(Tb + tq * Col8::GSTR + gq * 8 + k) = make_double2(Tn[k], Tn[k + 1]);
    };

    {
        double Gn[4][2], Tn[8];
        // prologue: T(0) and G(1)
        gram4(wbase, Gn);
        store_g(Gn);
        __syncwarp();
        trec(wbase + Col8::BETA, Tn);
        gram4(wbase + Col8::MAT, Gn);
        __syncwarp();
        store_t(Ts, Tn);
        store_g(Gn);
        __syncwarp();

#pragma unroll 1
        for (int mi = 0; mi < 4; ++mi) {
            const double* vb = wbase + mi * Col8::MAT;
            const double* Tb = Ts + (mi & 1) * 4 * Col8::GSTR;
            // next matrices (indices wrap on the last iterations: harmless extra work, keeps the loop body branch-free)
            trec(wbase + ((mi + 1) & 3) * Col8::MAT + Col8::BETA, Tn);
            gram4(wbase + ((mi + 2) & 3) * Col8::MAT, Gn);

            // ---- backward accumulation of matrix mi
            double qt[4][4][2];
#pragma unroll
            for (int cb = 0; cb < 4; ++cb)
#pragma unroll
                for (int rb = 0; rb < 4; ++rb) {
                    qt[cb][rb][0] = (cb == rb && 2 * tq == gq) ? 1.0 : 0.0;
                    qt[cb][rb][1] = (cb == rb && 2 * tq + 1 == gq) ? 1.0 : 0.0;
                }
#pragma unroll
            for (int p = 3; p >= 0; --p) {
                double f3[4][2], f1[4][2], w[4][2], w2[4][2];
#pragma unroll
                for (int rb = p; rb < 4; ++rb) {
                    f3[rb][0] = F3(vb, p, rb, 0);
                    f3[rb][1] = F3(vb, p, rb, 1);
                    if (rb > p) {
                        const double2 f = F1(vb, p, rb);
                        f1[rb][0] = f.x;
                        f1[rb][1] = f.y;
                    }
                }
                const double2 tt = *reinterpret_cast<const double2*>(Tb + p * Col8::GSTR + gq * 8 + 2 * tq);
                w[p][0] = f3[p][0];
                w[p][1] = f3[p][1];
#pragma unroll
                for (int cb = p + 1; cb < 4; ++cb) w[cb][0] = w[cb][1] = 0.0;
#pragma unroll
                for (int rb = p + 1; rb < 4; ++rb)
#pragma unroll
                    for (int i = 0; i < 2; ++i)
#pragma unroll
                        for (int cb = p + 1; cb < 4; ++cb) dmma_8x8x4(w[cb], qt[cb][rb][i], f1[rb][i]);
#pragma unroll
                for (int cb = p; cb < 4; ++cb) w2[cb][0] = w2[cb][1] = 0.0;
#pragma unroll
                for (int cb = p; cb < 4; ++cb) dmma_8x8x4(w2[cb], w[cb][0], tt.x);
#pragma unroll
                for (int cb = p; cb < 4; ++cb) dmma_8x8x4(w2[cb], w[cb][1], tt.y);
#pragma unroll
                for (int i = 0; i < 2; ++i)
#pragma unroll
                    for (int cb = p; cb < 4; ++cb)
#pragma unroll
                        for (int rb = p; rb < 4; ++rb) dmma_8x8x4(qt[cb][rb], w2[cb][i], f3[rb][i]);
            }

            const long long mat = mat0 + mi;
            if (mat < batch) {
                double* Qg = Q + mat * (N * N) + (2 * tq) * N + gq;
#pragma unroll
                for (int rb = 0; rb < 4; ++rb)
#pragma unroll
                    for (int i = 0; i < 2; ++i)
#pragma unroll
                        for (int cb = 0; cb < 4; ++cb) st_stream(Qg + (8 * rb + i) * N + 8 * cb, qt[cb][rb][i]);
            }
            __syncwarp();  // every lane has read G (for T(mi+1)) and -T(mi)
            store_t(Ts + ((mi + 1) & 1) * 4 * Col8::GSTR, Tn);
            store_g(Gn);
            __syncwarp();
        }
    }
}

}  // namespace lq

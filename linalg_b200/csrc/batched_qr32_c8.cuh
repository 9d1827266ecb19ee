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
//            After its own step a lane keeps its reflector v_c in registers (the diagonal of R on the side) and is no
//            longer updated, so the dot product v_j^T a_c that the later steps of the panel compute in that lane is the
//            Gram entry G_p[c][j] = v_c^T v_j: at the end of the panel lane c stores row c of G_p, which costs no
//            extra product.
//   storage  reflector j = rows (j & ~1)..31 in natural order, pivot patched to v0 (the row above an odd pivot to 0)
//            after the scalar chain, then beta, then the upper triangles of G_p (replaced by -T_p in the Q phase):
//            544 + 32 + 4 x 40 doubles per matrix.  Above 196 KB of shared memory per CTA the SM switches to a larger
//            carve-out and the R phase's streaming loads lose L1: an unpacked 8 x 8 layout (211 KB) costs more than the
//            Gram products it saves (profiles/r3_hh32_gram_from_steps.md).
//   Q phase  compact-WY on DMMA.8x8x4, one matrix at a time on all 32 lanes: Q^T lives in 16 accumulator tiles
//            (32 doubles / lane).  A DMMA.8x8x4 (the only f64 MMA shape sm_100a has; every mma.sync f64 shape lowers to
//            it) does 256 FMAs for one issue slot (the round-1 kernel's rank-1 DFMA Q phase issued ~1 930 FP64 instructions
//            per matrix).
//            T_p by the dlarft row recurrence from G_p, lane (g, t) = row g of panel t   ~36 DFMA for all four panels
//            for p = 3..0:  W^T = Q^T V_p ; W2^T = W^T (-T_p)^T ; Q^T += W2^T V_p^T   28 + 20 + 60 DMMA
//            An accumulator fragment IS a valid A operand when the contraction index is permuted (k = t <-> column
//            2t+i), so W^T and W2^T never leave registers; V is read from shared memory directly in B-fragment order.
//
// Tile / fragment conventions (lane l, g = l >> 2, t = l & 3), mma.m8n8k4.f64:
//   A[g][t], B[t][g], C[g][2t], C[g][2t+1].
//   qt[cb][rb][i] = Q[8 rb + 2t + i][8 cb + g]          (tile (cb, rb) of Q^T)
//   F1(p, rb, i)  = V[8 rb + 2t + i][8 p + g]           (B operand of W^T = Q^T V)
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
    // upper triangle of an 8 x 8 block (G_p, then -T_p) in column pairs: row r keeps the pairs q = r/2..3 (40 doubles);
    // tpos(r, q) is the offset of the pair (2q, 2q + 1) of row r
    __host__ __device__ static constexpr int tpos(int r, int q) {
        return 2 * (8 * (r >> 1) - (r >> 1) * ((r >> 1) - 1) + (r & 1) * (4 - (r >> 1)) + q - (r >> 1));
    }
    static constexpr int VDOUBLES = 544;
    static constexpr int BETA = VDOUBLES;  // beta_j, read by the apply steps of the later panels
    static constexpr int TOFF = BETA + 32; // G_p of the four panels (tpos layout), overwritten by -T_p in the Q phase
    static constexpr int TSTR = 42;        // 21 16-byte words: the four panels read by one instruction of the T recurrence
                                           // start in four different bank quads
    static constexpr int MAT = TOFF + 3 * TSTR + 40 + 6;  // 374 16-byte words = 6 (mod 8): the four matrices of a warp hit
                                                          // four different bank quads.  4 MAT doubles per warp keep the
                                                          // 8-warp CTA within the 196 KB shared-memory carve-out
    static constexpr int WARP_DOUBLES = 4 * MAT;
};
static_assert(Col8::tpos(7, 3) == 38 && Col8::tpos(6, 3) == 36 && Col8::tpos(2, 1) == 16, "packed triangle");
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
        int tw[4];  // where lane c writes its row of the panel's G
#pragma unroll
        for (int q = 0; q < 4; ++q) tw[q] = Col8::TOFF + Col8::tpos(c, q);

#pragma unroll
        for (int p = 0; p < 4; ++p) {
            const int col = 8 * p + c;
            double a[N];
            double rdiag = 0.0;        // R[col][col]; after its own step the lane keeps v_col in a[col..31]
            double grow[8];            // grow[k] = G_p[c][k] = v_c^T v_k for k > c
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

                // v^T a_c = x^T a_c + alpha * a[j][c].  A finished lane (c < jj) holds v_c from row j on, so there it is
                // the Gram entry G[c][jj]; only the lanes right of the pivot are updated.
                const double vta = fma(alpha, a[j], dot);
                grow[jj] = vta;
                const double s = c > jj ? beta * vta : 0.0;

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
                // the owner keeps its reflector (pivot v0) and the diagonal of R on the side; the skipped column keeps x0
                if (c == jj) {
                    rdiag = skip ? a[j] : -alpha;
                    a[j] = v0;
                }
            }

            // ---- row c of G_p to shared memory (the entries left of and on the diagonal are never read)
#pragma unroll
            for (int q = 0; q < 4; ++q)
                if (q >= (c >> 1))
                    *reinterpret_cast<double2*>(vb + Col8::TSTR * p + tw[q]) = make_double2(grow[2 * q], grow[2 * q + 1]);
            __syncwarp();  // the last pivot patch of this panel is visible to the apply steps of the next one

            // ---- store the R columns of this panel (strict lower triangle forced to exact zeros, qr.py:97)
            if (valid) {
                double* Rg = R + mat * (N * N) + col;
#pragma unroll
                for (int i = 0; i < N; ++i) {
                    double v = a[i];
                    if (i >= 8 * p + 8) v = 0.0;
                    else if (i >= 8 * p) v = (i < col) ? v : (i == col ? rdiag : 0.0);
                    st_stream(Rg + i * N, v);
                }
            }
        }
    }
    __syncwarp();  // the reflectors and G of every panel are visible to the Q phase

    // ================= Q phase: Q = (I - V0 T0 V0^T) ... (I - V3 T3 V3^T), backward accumulation on DMMA ==========
    // Fragment conventions as in the header comment (g = gq, t = tq).  Software-pipelined over the four matrices of the
    // warp: while the block reflectors of matrix mi are applied (DMMA chains), the T recurrence of matrix mi+1 (a DFMA
    // chain) runs in the same instruction stream and fills the bubbles.
    const int gq = lane >> 2, tq = lane & 3;
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
    const int tro = Col8::TOFF + Col8::tpos(gq, tq);  // -T_p[g][2t + i] at tro + TSTR p
    const bool tup = tq >= (gq >> 1);                  // the pair is stored (the lower triangle of -T is zero)
    int two[4];                                        // row g of panel t, pair q (the T recurrence)
#pragma unroll
    for (int q = 0; q < 4; ++q) two[q] = Col8::TOFF + Col8::TSTR * tq + Col8::tpos(gq, q);
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

    // -T of panel tq, row gq (dlarft, forward / columnwise): T[g][k] = -beta_k sum_{m=g}^{k-1} T[g][m] G[m][k]
    auto trec = [&](const double* vb, double (&Tn)[8]) {
        const double* G = vb + Col8::TOFF + Col8::TSTR * tq;
        double bk[8], acc[8];
#pragma unroll
        for (int k = 0; k < 8; k += 2) {
            const double2 b2 = *reinterpret_cast<const double2*>(vb + Col8::BETA + 8 * tq + k);
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
                    const double2 g2 = *reinterpret_cast<const double2*>(G + Col8::tpos(k, kk >> 1));
                    if (kk > k) acc[kk] = fma(tk, g2.x, acc[kk]);
                    acc[kk + 1] = fma(tk, g2.y, acc[kk + 1]);
                }
            }
        }
    };
    // -T replaces G in place, once every lane has read G
    auto store_t = [&](double* vb, const double (&Tn)[8]) {
#pragma unroll
        for (int q = 0; q < 4; ++q)
            if (q >= (gq >> 1)) *reinterpret_cast<double2*>(vb + two[q]) = make_double2(Tn[2 * q], Tn[2 * q + 1]);
    };

    double Tn[8];
    trec(wbase, Tn);
    __syncwarp();
    store_t(wbase, Tn);
    __syncwarp();

#pragma unroll 1
    for (int mi = 0; mi < 4; ++mi) {
        const double* vb = wbase + mi * Col8::MAT;
        // next matrix (wraps to matrix 0 on the last iteration, whose -T is no longer read: harmless extra work, keeps
        // the loop body branch-free)
        double* nb = wbase + ((mi + 1) & 3) * Col8::MAT;
        trec(nb, Tn);

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
            double2 tt = make_double2(0.0, 0.0);
            if (tup) tt = *reinterpret_cast<const double2*>(vb + tro + Col8::TSTR * p);
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
        __syncwarp();  // every lane has read G of matrix mi+1 and -T of matrix mi
        store_t(nb, Tn);
        __syncwarp();
    }
}

}  // namespace lq

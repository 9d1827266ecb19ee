// K3 (round 2): batched Householder least squares, ONE WARP PER SYSTEM, block reflectors on the FP64 tensor pipe.
//
// Reference semantics: linalg/qr.py:122-134 (least_squares_householder_qr: x = R^-1 (Q^T b)) and, for the MGS entry point
// linalg/qr.py:103-119 (least_squares_qr), the same solution plus the "R[j, j] < EPS" dependence test of linalg/qr.py:40-41
// (|R[j, j]| is the same number for every QR factorisation of A).  Only X is observable through these entry points, so the
// kernel is free to choose its reflectors: it streams [A | B] through registers in blocks of 32 rows and folds each block
// into the running triangle with a "triangle on top of a dense block" Householder step (the structure of LAPACK's
// dtpqrt2): reflector j of a step is v = [v0 e_j ; x], x = column j of the block, so only ROW j of R and the block change.
// Q is never formed, A and B are read exactly once, nothing but X is written.
//
// Round 1 ran this scheme as a CTA-wide column loop (256 steps per system, a block barrier and an 80-column rank-1 update on
// DFMA in every step, ~1 us per step: 13 % of the FP64 peak).  Here:
//   * the block lives in registers as TRANSPOSED 8 x 8 tiles in the accumulator layout of mma.sync.m8n8k4.f64
//     (lane (g, t) of tile (cb, rb): column 8 cb + g, rows 8 rb + 2 t + {0, 1}).  An accumulator register is at the same
//     time a valid A operand of the next product (the k index may be permuted: {0,2,4,6} | {1,3,5,7}), so
//         W^T  = R_p^T D + C^T X          (8 DMMA per tile, both operands straight from registers)
//         W'^T = W^T (-T)                 (2 DMMA)
//         C^T += W'^T X^T,  R_p^T += W'^T D   (8 DMMA, X^T from shared memory)
//     need no shuffles, no layout changes and no shared-memory traffic for C;
//   * columns are factored 8 at a time (a panel): the scalar chain of a column step touches 8 columns instead of 80, and
//     there is no block-wide barrier anywhere -- a warp only ever synchronises with itself;
//   * T comes from the Gram matrix X^T X (the top parts of the reflectors are disjoint unit vectors and do not
//     contribute off the diagonal); its column k falls out of column step k's dot products and is consumed during
//     step k + 1, off the critical chain.
// R^T (36 upper-triangular tiles), the 64 x 16 right-hand-side rows (16 tiles) and 2.2 KB of scratch live in shared memory:
// 28.9 KB per warp, 8 warps per SM (the register file allows no more at 255 registers: a 32 x 80 block is 160 of them).
#pragma once

#include <type_traits>

#include "common.cuh"

namespace lq {

struct LsTile {
    static constexpr int NCB = 8;   // column blocks of A (n <= 64)
    static constexpr int NRT = 2;   // right-hand-side tiles (nrhs <= 16)
    static constexpr int RB = 4;    // 8-row blocks per streamed block
    static constexpr int ROWS = 8 * RB;
    // tile (cb, p) of R^T, p <= cb < 8: row panel p of R holds the tiles cb = p .. 7
    __host__ __device__ static constexpr int tile(int cb, int p) { return 8 * p - (p * (p - 1)) / 2 + (cb - p); }
    static constexpr int A_TILES = 36;
    static constexpr int Y_TILE0 = A_TILES;                 // y tile (rt, p) at Y_TILE0 + 8 * rt + p
    static constexpr int XS = (A_TILES + 8 * NRT) * 64;     // 32 rows x 8: the panel's reflectors, row-major, XOR-swizzled
                                                            // (element (r, c) at 8 r + (c ^ 2 ((r >> 1) & 3)): the column
                                                            // publishes / reads and the 128-bit row reads are conflict free);
                                                            // its first 64 doubles are reused for -T once X^T is in registers,
                                                            // and as the scratch of the back-substitution
    static constexpr int GS = XS + ROWS * 8;                // 2 x 8: column k of the Gram matrix X^T X (double buffered)
    static constexpr int DV = GS + 16;                      // 8: v0 of the panel's reflectors
    static constexpr int WARP_DOUBLES = DV + 8;             // 3608 doubles = 28 864 B: eight warps per SM
};
static_assert(LsTile::tile(7, 7) == 35, "packed triangle");

// info_mode: 0 = none, 1 = MGS semantics (first column with |R[j, j]| < 1e-12, linalg/qr.py:40-41, 1-based),
//            2 = exactly singular R (np.linalg.solve raises LinAlgError there, linalg/qr.py:134)
template <int WARPS, int MINB>
__global__ void __launch_bounds__(WARPS * 32, MINB)
    lstsq_tile_kernel(const double* __restrict__ A, const double* __restrict__ B, double* __restrict__ X, int* __restrict__ info,
                      long long batch, int m, int n, int nrhs, int info_mode) {
    using L = LsTile;
    constexpr int NCB = L::NCB, NRT = L::NRT, RB = L::RB;
    extern __shared__ __align__(16) double sm[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane >> 2, t = lane & 3;
    const long long sys = (long long)blockIdx.x * WARPS + warp;
    if (sys >= batch) return;  // warps never synchronise with each other

    double* Rt = sm + (size_t)warp * L::WARP_DOUBLES;
    double* Xs = Rt + L::XS;
    double* Ts = Xs;  // aliased: written only after the panel's X^T operands have been loaded
    double* Gs = Rt + L::GS;
    double* Dv = Rt + L::DV;

    const double* Ag = A + sys * (long long)m * n;
    const double* Bg = B + sys * (long long)m * nrhs;
    const int npan = (n + 7) >> 3;
    const bool full_cols = (n == 8 * NCB) && (nrhs == 8 * NRT);

    {
        const double2 z = make_double2(0.0, 0.0);
        for (int e = lane; e < L::XS / 2; e += 32) reinterpret_cast<double2*>(Rt)[e] = z;
    }
    __syncwarp();

    for (int r0 = 0; r0 < m; r0 += L::ROWS) {
        // ---- the next 32 rows of [A | B] as transposed accumulator tiles
        double ct[NCB + NRT][RB][2];
        if (r0 + L::ROWS < m) {
            // the block after this one: into L2 now, so that its loads are short-latency hits when the panel loop is done
            const long long a0 = (long long)(r0 + L::ROWS) * n * 8, a1 = min((long long)(r0 + 2 * L::ROWS), (long long)m) * n * 8;
            for (long long off = a0 + (long long)lane * 128; off < a1; off += 32 * 128)
                asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const char*>(Ag) + off));
            const long long b0 = (long long)(r0 + L::ROWS) * nrhs * 8, b1 = min((long long)(r0 + 2 * L::ROWS), (long long)m) * nrhs * 8;
            for (long long off = b0 + (long long)lane * 128; off < b1; off += 32 * 128)
                asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const char*>(Bg) + off));
        }
        if (full_cols && r0 + L::ROWS <= m) {
#pragma unroll
            for (int rb = 0; rb < RB; ++rb)
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const long long row = r0 + 8 * rb + 2 * t + e;
#pragma unroll
                    for (int cb = 0; cb < NCB; ++cb) ct[cb][rb][e] = ld_stream(Ag + row * (8 * NCB) + 8 * cb + g);
#pragma unroll
                    for (int rt = 0; rt < NRT; ++rt) ct[NCB + rt][rb][e] = ld_stream(Bg + row * (8 * NRT) + 8 * rt + g);
                }
        } else {
#pragma unroll
            for (int rb = 0; rb < RB; ++rb)
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const long long row = r0 + 8 * rb + 2 * t + e;
                    const bool rok = row < m;
#pragma unroll
                    for (int cb = 0; cb < NCB; ++cb)
                        ct[cb][rb][e] = (rok && 8 * cb + g < n) ? ld_stream(Ag + row * n + 8 * cb + g) : 0.0;
#pragma unroll
                    for (int rt = 0; rt < NRT; ++rt)
                        ct[NCB + rt][rb][e] = (rok && 8 * rt + g < nrhs) ? ld_stream(Bg + row * nrhs + 8 * rt + g) : 0.0;
                }
        }

#pragma unroll 1
        for (int p = 0; p < npan; ++p) {
            // ---- the panel tile (column block p of the block)
            double P[RB][2];
#pragma unroll
            for (int cb = 0; cb < NCB; ++cb)
                if (cb == p) {
#pragma unroll
                    for (int rb = 0; rb < RB; ++rb) P[rb][0] = ct[cb][rb][0], P[rb][1] = ct[cb][rb][1];
                }
            double* rpp = Rt + L::tile(p, p) * 64;  // diagonal tile of R^T: [c][i] = R[8p + i][8p + c]
            double* xrow = Xs + (2 * t) * 8;        // + 64 rb (+ 8): rows 8 rb + 2 t (+ 1) of the published reflectors; their swizzle is 2 t

            // ---- factor the 8 columns of [R_pp ; P].  T (dlarft, forward / columnwise) is built on the way, off the
            // critical chain: column k of the Gram matrix X^T X falls out of step k's dot products (lanes g < k), is
            // broadcast through shared memory and consumed during step k + 1:
            //     T[g][k] = -beta_k sum_{m = g}^{k - 1} T[g][m] G[m][k]
            double Trow[8];
            double beta_prev = 0.0;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                if (g == j) {
#pragma unroll
                    for (int rb = 0; rb < RB; ++rb) {
                        xrow[64 * rb + (j ^ (2 * t))] = P[rb][0];
                        xrow[64 * rb + 8 + (j ^ (2 * t))] = P[rb][1];
                    }
                }
                const double rjc = rpp[g * 8 + j];  // R[j][c = g]
                const double x0 = rpp[j * 8 + j];
                __syncwarp();
                double xk[RB][2];
                double d0 = 0.0, d1 = 0.0, q0 = 0.0, q1 = 0.0;
#pragma unroll
                for (int rb = 0; rb < RB; ++rb) {
                    xk[rb][0] = xrow[64 * rb + (j ^ (2 * t))];
                    xk[rb][1] = xrow[64 * rb + 8 + (j ^ (2 * t))];
                    d0 = fma(xk[rb][0], P[rb][0], d0);
                    d1 = fma(xk[rb][1], P[rb][1], d1);
                    q0 = fma(xk[rb][0], xk[rb][0], q0);
                    q1 = fma(xk[rb][1], xk[rb][1], q1);
                }
                double d = d0 + d1, q = q0 + q1;
                d += __shfl_xor_sync(0xffffffffu, d, 1);
                q += __shfl_xor_sync(0xffffffffu, q, 1);
                d += __shfl_xor_sync(0xffffffffu, d, 2);  // x^T a_c for c = g
                q += __shfl_xor_sync(0xffffffffu, q, 2);  // x^T x

                // column j - 1 of T (needs G[.][j - 1], published in the previous step, and beta_{j-1})
                if (j > 0) {
                    const double* gk = Gs + ((j - 1) & 1) * 8;
                    double a0 = 0.0, a1 = 0.0;
#pragma unroll
                    for (int mm = 0; mm < j - 1; ++mm) {
                        if (mm & 1) a1 = fma(Trow[mm], gk[mm], a1);
                        else a0 = fma(Trow[mm], gk[mm], a0);
                    }
                    const double sel = (g == j - 1) ? 1.0 : 0.0, lt = (g < j - 1) ? 1.0 : 0.0;
                    Trow[j - 1] = beta_prev * fma(-lt, a0 + a1, sel);
                }
                if (t == 0 && g < j) Gs[(j & 1) * 8 + g] = d;

                const double ss = fma(x0, x0, q);
                const double ssc = ss + 1e-300;
                // y = 1 / ||[x0 ; x]||, beta = 2 / v^T v = y^2 / (1 + |x0| y); the reciprocal is seeded from the UNREFINED y
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
                // skip only an exactly zero column: this block holds part of the column, and the rows of a skipped
                // block would be lost (see stream_factor_block); |R_jj| ends as the full remaining norm, which the
                // report below compares with 1e-12 (MGS) or 0 (Householder)
                const bool skip = ss == 0.0;
                const double alpha = copysign(nrm, x0);
                const double v0 = skip ? 0.0 : x0 + alpha;
                const double beta = skip ? 0.0 : (y * y) * u;
                beta_prev = beta;

                const double s = (g > j) ? beta * fma(v0, rjc, d) : 0.0;
                {
                    const double val = (g > j) ? fma(-s, v0, rjc) : -alpha;
                    if (t == 0 && (g > j || (g == j && !skip))) rpp[g * 8 + j] = val;
                }
                if (lane == 0) Dv[j] = v0;
#pragma unroll
                for (int rb = 0; rb < RB; ++rb) {
                    P[rb][0] = fma(-s, xk[rb][0], P[rb][0]);
                    P[rb][1] = fma(-s, xk[rb][1], P[rb][1]);
                }
            }
            // X^T operands of the update (row 8 rb + g, columns 2 t, 2 t + 1), the last column of T, then -T row g to shared
            // memory (B operands need it transposed) -- into the space of X, which is in registers by then
            __syncwarp();
            double2 Xt[RB];
#pragma unroll
            for (int rb = 0; rb < RB; ++rb)
                Xt[rb] = *reinterpret_cast<const double2*>(Xs + (8 * rb + g) * 8 + ((2 * t) ^ (2 * ((g >> 1) & 3))));
            const double2 d2 = *reinterpret_cast<const double2*>(Dv + 2 * t);
            {
                const double* gk = Gs + 8;
                double a0 = 0.0, a1 = 0.0;
#pragma unroll
                for (int mm = 0; mm < 7; ++mm) {
                    if (mm & 1) a1 = fma(Trow[mm], gk[mm], a1);
                    else a0 = fma(Trow[mm], gk[mm], a0);
                }
                const double sel = (g == 7) ? 1.0 : 0.0, lt = (g < 7) ? 1.0 : 0.0;
                Trow[7] = beta_prev * fma(-lt, a0 + a1, sel);
            }
            __syncwarp();  // every lane holds its X^T operands: the space takes -T
            if (t == 0) {
#pragma unroll
                for (int k = 0; k < 8; k += 2) *reinterpret_cast<double2*>(Ts + g * 8 + k) = make_double2(-Trow[k], -Trow[k + 1]);
            }
            __syncwarp();
            const double nT0 = Ts[(2 * t) * 8 + g], nT1 = Ts[(2 * t + 1) * 8 + g];

            // ---- block reflector on the trailing column blocks and the right-hand sides, up to three tiles at a time (the
            // accumulator chains of the tiles of a group interleave; NT is a compile-time count, so a group never
            // computes a tile left of the panel)
            auto apply = [&](auto nt_tag, double* ta, double (&ca)[RB][2], double* tb, double (&cbk)[RB][2], double* tc, double (&cc)[RB][2]) {
                constexpr int NT = decltype(nt_tag)::value;
                double2 ra = *reinterpret_cast<const double2*>(ta + g * 8 + 2 * t), rb2 = ra, rc = ra;
                if (NT > 1) rb2 = *reinterpret_cast<const double2*>(tb + g * 8 + 2 * t);
                if (NT > 2) rc = *reinterpret_cast<const double2*>(tc + g * 8 + 2 * t);
                double wa[2] = {ra.x * d2.x, ra.y * d2.y}, wa2[2] = {0.0, 0.0};
                double wb[2] = {rb2.x * d2.x, rb2.y * d2.y}, wb2[2] = {0.0, 0.0};
                double wc[2] = {rc.x * d2.x, rc.y * d2.y}, wc2[2] = {0.0, 0.0};
#pragma unroll
                for (int rb = 0; rb < RB; rb += 2)
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        dmma_8x8x4(wa, ca[rb][e], P[rb][e]);
                        if (NT > 1) dmma_8x8x4(wb, cbk[rb][e], P[rb][e]);
                        if (NT > 2) dmma_8x8x4(wc, cc[rb][e], P[rb][e]);
                        dmma_8x8x4(wa2, ca[rb + 1][e], P[rb + 1][e]);
                        if (NT > 1) dmma_8x8x4(wb2, cbk[rb + 1][e], P[rb + 1][e]);
                        if (NT > 2) dmma_8x8x4(wc2, cc[rb + 1][e], P[rb + 1][e]);
                    }
                wa[0] += wa2[0], wa[1] += wa2[1];
                wb[0] += wb2[0], wb[1] += wb2[1];
                wc[0] += wc2[0], wc[1] += wc2[1];
                double za[2] = {0.0, 0.0}, zb[2] = {0.0, 0.0}, zc[2] = {0.0, 0.0};
                dmma_8x8x4(za, wa[0], nT0);
                if (NT > 1) dmma_8x8x4(zb, wb[0], nT0);
                if (NT > 2) dmma_8x8x4(zc, wc[0], nT0);
                dmma_8x8x4(za, wa[1], nT1);
                if (NT > 1) dmma_8x8x4(zb, wb[1], nT1);
                if (NT > 2) dmma_8x8x4(zc, wc[1], nT1);
#pragma unroll
                for (int rb = 0; rb < RB; ++rb) {
                    dmma_8x8x4(ca[rb], za[0], Xt[rb].x);
                    if (NT > 1) dmma_8x8x4(cbk[rb], zb[0], Xt[rb].x);
                    if (NT > 2) dmma_8x8x4(cc[rb], zc[0], Xt[rb].x);
                }
#pragma unroll
                for (int rb = 0; rb < RB; ++rb) {
                    dmma_8x8x4(ca[rb], za[1], Xt[rb].y);
                    if (NT > 1) dmma_8x8x4(cbk[rb], zb[1], Xt[rb].y);
                    if (NT > 2) dmma_8x8x4(cc[rb], zc[1], Xt[rb].y);
                }
                ra.x = fma(za[0], d2.x, ra.x), ra.y = fma(za[1], d2.y, ra.y);
                *reinterpret_cast<double2*>(ta + g * 8 + 2 * t) = ra;
                if (NT > 1) {
                    rb2.x = fma(zb[0], d2.x, rb2.x), rb2.y = fma(zb[1], d2.y, rb2.y);
                    *reinterpret_cast<double2*>(tb + g * 8 + 2 * t) = rb2;
                }
                if (NT > 2) {
                    rc.x = fma(zc[0], d2.x, rc.x), rc.y = fma(zc[1], d2.y, rc.y);
                    *reinterpret_cast<double2*>(tc + g * 8 + 2 * t) = rc;
                }
            };
            using N1 = std::integral_constant<int, 1>;
            using N2 = std::integral_constant<int, 2>;
            using N3 = std::integral_constant<int, 3>;
            auto taddr = [&](int cb) -> double* { return Rt + L::tile(cb, p) * 64; };
            double* y0 = Rt + (L::Y_TILE0 + p) * 64;
            double* y1 = Rt + (L::Y_TILE0 + 8 + p) * 64;
            // groups: {rhs 0, rhs 1, 7}, {6, 5, 4}, {3, 2, 1}; the column blocks of a group that lie right of the panel
            if (p < 7) apply(N3{}, y0, ct[NCB], y1, ct[NCB + 1], taddr(7), ct[7]);
            else apply(N2{}, y0, ct[NCB], y1, ct[NCB + 1], y1, ct[NCB + 1]);
            if (p < 4) apply(N3{}, taddr(6), ct[6], taddr(5), ct[5], taddr(4), ct[4]);
            else if (p == 4) apply(N2{}, taddr(6), ct[6], taddr(5), ct[5], taddr(5), ct[5]);
            else if (p == 5) apply(N1{}, taddr(6), ct[6], taddr(6), ct[6], taddr(6), ct[6]);
            if (p < 1) apply(N3{}, taddr(3), ct[3], taddr(2), ct[2], taddr(1), ct[1]);
            else if (p == 1) apply(N2{}, taddr(3), ct[3], taddr(2), ct[2], taddr(2), ct[2]);
            else if (p == 2) apply(N1{}, taddr(3), ct[3], taddr(3), ct[3], taddr(3), ct[3]);
            __syncwarp();
        }
    }

    // ---- dependence / singularity report from the diagonal of R
    if (info != nullptr) {
        int first = 0x7fffffff;
        for (int j = lane; j < n; j += 32) {
            const double rjj = fabs(Rt[L::tile(j >> 3, j >> 3) * 64 + (j & 7) * 9]);
            const bool bad = (info_mode == 1) ? (rjj < kEps) : (rjj == 0.0);
            if (bad) first = min(first, j + 1);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) first = min(first, __shfl_xor_sync(0xffffffffu, first, o));
        if (lane == 0) info[sys] = (first == 0x7fffffff) ? 0 : first;
    }

    // ---- back-substitution R X = Y on transposed tiles: X^T[ib] = (Y^T[ib] - sum_{jb > ib} X^T[jb] R[ib][jb]^T) R[ib][ib]^-T
    double xt[NRT][8][2];
#pragma unroll
    for (int rt = 0; rt < NRT; ++rt)
#pragma unroll
        for (int ib = 0; ib < 8; ++ib) xt[rt][ib][0] = xt[rt][ib][1] = 0.0;
#pragma unroll
    for (int ib = 7; ib >= 0; --ib) {
        if (ib < npan) {
#pragma unroll
            for (int rt = 0; rt < NRT; ++rt) {
                const double2 y2 = *reinterpret_cast<const double2*>(Rt + (L::Y_TILE0 + 8 * rt + ib) * 64 + g * 8 + 2 * t);
                xt[rt][ib][0] = y2.x;
                xt[rt][ib][1] = y2.y;
            }
#pragma unroll
            for (int jb = 7; jb > ib; --jb) {
                if (jb < npan) {
                    const double* tl = Rt + L::tile(jb, ib) * 64;  // [c = j][i]
                    const double b0 = -tl[(2 * t) * 8 + g], b1 = -tl[(2 * t + 1) * 8 + g];
#pragma unroll
                    for (int rt = 0; rt < NRT; ++rt) {
                        dmma_8x8x4(xt[rt][ib], xt[rt][jb][0], b0);
                        dmma_8x8x4(xt[rt][ib], xt[rt][jb][1], b1);
                    }
                }
            }
            // diagonal block: lane l solves right-hand side (l & 15) against the 8 x 8 triangle (lanes 16 .. 31 mirror 0 .. 15)
            __syncwarp();
#pragma unroll
            for (int rt = 0; rt < NRT; ++rt)
                *reinterpret_cast<double2*>(Xs + rt * 64 + g * 8 + 2 * t) = make_double2(xt[rt][ib][0], xt[rt][ib][1]);
            const double* dt = Rt + L::tile(ib, ib) * 64;  // R[i][j] = dt[j * 8 + i]
            const double rd = dt[(lane & 7) * 9];
            const double rinv_l = (8 * ib + (lane & 7) < n) ? 1.0 / rd : 0.0;
            __syncwarp();
            double z[8];
            {
                const double* zs = Xs + (lane & 15) * 8;
#pragma unroll
                for (int i = 0; i < 8; i += 2) {
                    const double2 z2 = *reinterpret_cast<const double2*>(zs + i);
                    z[i] = z2.x;
                    z[i + 1] = z2.y;
                }
            }
#pragma unroll
            for (int i = 7; i >= 0; --i) {
                double acc = z[i];
#pragma unroll
                for (int j = i + 1; j < 8; ++j) acc = fma(-dt[j * 8 + i], z[j], acc);
                z[i] = acc * __shfl_sync(0xffffffffu, rinv_l, i);
            }
            __syncwarp();
            if (lane < 16) {
                double* zs = Xs + lane * 8;
#pragma unroll
                for (int i = 0; i < 8; i += 2) *reinterpret_cast<double2*>(zs + i) = make_double2(z[i], z[i + 1]);
            }
            __syncwarp();
#pragma unroll
            for (int rt = 0; rt < NRT; ++rt) {
                const double2 x2 = *reinterpret_cast<const double2*>(Xs + rt * 64 + g * 8 + 2 * t);
                xt[rt][ib][0] = x2.x;
                xt[rt][ib][1] = x2.y;
            }
        }
    }

    double* Xg = X + sys * (long long)n * nrhs;
#pragma unroll
    for (int ib = 0; ib < 8; ++ib)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int i = 8 * ib + 2 * t + e;
#pragma unroll
            for (int rt = 0; rt < NRT; ++rt) {
                const int k = 8 * rt + g;
                if (i < n && k < nrhs) st_stream(Xg + (long long)i * nrhs + k, xt[rt][ib][e]);
            }
        }
}

}  // namespace lq

// Batched economy SVD on the A^T A route (linalg/svd.py:10-82) for m >= n, n <= 32, m <= SvdSmall::M_SMALL: one warp
// per matrix, everything the single-matrix pipeline (svd_gram_local) does in one launch.
//
//   Gram   G = A^T A: A streams through the warp's staging buffer in contiguous tiles of whole rows (16-byte loads when
//          the tile is 16-byte aligned); lane j accumulates column j of G in 32 registers from broadcast reads of the row.
//          G is exactly symmetric (lane i and lane j form the same products in the same order), and a zero column of A
//          gives an exactly zero row and column of G.
//   Jacobi two-sided cyclic Jacobi on 2^-e G with max|diag| in [1, 2) (the scaling of jacobi_kernel: exact, so the
//          result scales bit for bit under powers of two), round-robin pairs (rr_pair), the rotation test of the single
//          path (|g_pq| > 4 eps sqrt(g_pp g_qq) and |g_pq| > eps^2 max|diag|), at most 40 sweeps.  G and V live in
//          warp-private shared memory with an odd pitch: in the column phase lane i updates row i of G and V, in the
//          row phase lane j updates column j of G (conflict-free both ways).  A round whose pair does not rotate is
//          skipped by the whole warp.  A zero row and column never rotates, so its eigenvalue stays exactly 0.
//   post   descending order by counting (NaN sorts first, ties by index, always a permutation), s = sqrt(max(lambda, 0)) with NaN kept,
//          rank = #(s > tol), Vt = V^T, U[:, j] = A (v_j / s_j) for s_j > tol and 0 otherwise: a second pass over A,
//          which is still in L2 (the matrices of all resident warps take ~15 MB).  U and Vt are written with streaming
//          stores so that they do not evict the A tiles of other warps.
// No register array is indexed at run time: the accumulators of the Gram and the column of V / s of the U pass are
// unrolled over 32 entries with a run-time guard.
#pragma once

#include "common.cuh"

namespace lq {

struct SvdSmall {
    static constexpr int NMAX = 32;          // columns (after transposition)
    static constexpr int M_SMALL = 4096;     // rows; taller matrices go through svd_gram_local one by one
    static constexpr int LD = NMAX + 1;      // odd pitch of G and V
    static constexpr int MAT = NMAX * LD;
    static constexpr int STAGE = 1024;       // doubles of A per tile; the tile buffer is V's storage (V is not live then)
    static constexpr int MAX_SWEEPS = 40;
    // G, V, 16 (c, s) pairs, 16 (p, q) pairs, 32 column sources
    static constexpr int WARP_DOUBLES = 2 * MAT + 32 + 16 + 16;
    static_assert(STAGE <= MAT, "the A tile lives in V's storage");
};

inline bool svd_small_supported(long long m, int n) { return n >= 1 && n <= SvdSmall::NMAX && m >= n && m <= SvdSmall::M_SMALL; }

template <int WARPS>
__global__ void __launch_bounds__(WARPS * 32) svd_small_kernel(const double* __restrict__ A, long long batch, int m, int n,
                                                               double tol, double* __restrict__ U, double* __restrict__ S,
                                                               double* __restrict__ Vt, int* __restrict__ rank) {
    using K = SvdSmall;
    constexpr unsigned FULL = 0xffffffffu;
    extern __shared__ __align__(16) double smem[];
    const int ln = threadIdx.x & 31;
    const long long b = (long long)blockIdx.x * WARPS + (threadIdx.x >> 5);
    if (b >= batch) return;  // warp-uniform; the kernel has no block barrier
    double* G = smem + (threadIdx.x >> 5) * K::WARP_DOUBLES;
    double* V = G + K::MAT;
    double* stage = V;
    double2* cs = reinterpret_cast<double2*>(V + K::MAT);
    int2* pq = reinterpret_cast<int2*>(cs + 16);
    int* src = reinterpret_cast<int*>(pq + 16);
    const double* Ab = A + b * (long long)m * n;
    const int rows_per_tile = (K::STAGE / n) & ~1;

    // rows [r0, r0 + rows) of A into the tile buffer (whole rows, contiguous in memory)
    auto load_tile = [&](int r0, int rows) {
        const double* g = Ab + (long long)r0 * n;
        const int cnt = rows * n;
        if ((reinterpret_cast<uintptr_t>(g) & 15) == 0) {
            for (int e = 2 * ln; e + 1 < cnt; e += 64)
                *reinterpret_cast<double2*>(stage + e) = __ldg(reinterpret_cast<const double2*>(g + e));
            if ((cnt & 1) && ln == 0) stage[cnt - 1] = __ldg(g + cnt - 1);
        } else {
            for (int e = ln; e < cnt; e += 32) stage[e] = __ldg(g + e);
        }
        __syncwarp();
    };

    // ---- G = A^T A, lane j owns column j
    {
        double g[K::NMAX];
#pragma unroll
        for (int i = 0; i < K::NMAX; ++i) g[i] = 0.0;
        for (int r0 = 0; r0 < m; r0 += rows_per_tile) {
            const int rows = min(rows_per_tile, m - r0);
            load_tile(r0, rows);
            for (int r = 0; r < rows; ++r) {
                const double* row = stage + r * n;
                const double aj = ln < n ? row[ln] : 0.0;
#pragma unroll
                for (int i = 0; i < K::NMAX; ++i)
                    if (i < n) g[i] = fma(row[i], aj, g[i]);
            }
            __syncwarp();
        }
        bool bad = false;
#pragma unroll
        for (int i = 0; i < K::NMAX; ++i) {
            G[i * K::LD + ln] = g[i];  // rows / columns >= n are exactly 0 (for finite A)
            bad |= i < n && !isfinite(g[i]);
        }
        // a NaN or infinite entry of G: no sweep and every eigenvalue NaN, as jacobi_kernel / jacobi1s_kernel do (so this
        // route agrees with the single-matrix route on non-finite input)
        const bool nonfinite = __any_sync(FULL, ln < n && bad);
        __syncwarp();
        // work on 2^-e G with max|diag| in [1, 2), exactly as jacobi_kernel does; lambda is scaled back by 2^e below
        double d = ln < n ? fabs(G[ln * K::LD + ln]) : 0.0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) d = fmax(d, __shfl_xor_sync(FULL, d, o));
        const int e = (d > 0.0 && isfinite(d)) ? ilogb(d) : 0;
        if (e != 0) {
#pragma unroll
            for (int i = 0; i < K::NMAX; ++i) G[i * K::LD + ln] = scalbn(g[i], -e);
        }
#pragma unroll
        for (int i = 0; i < K::NMAX; ++i) V[i * K::LD + ln] = i == ln ? 1.0 : 0.0;
        __syncwarp();

        const double floor_abs = 4.9303806576313238e-32 * scalbn(d, -e);  // eps^2 * max|diag|
        const double rel_tol = 4.0 * 1.1102230246251565e-16;
        const int ne = (n + 1) & ~1, half = ne / 2;
        for (int sweep = 0; sweep < (nonfinite ? 0 : K::MAX_SWEEPS); ++sweep) {
            bool rotated = false;
            for (int rd = 0; rd < ne - 1; ++rd) {
                if (ln < half) {
                    int p, q;
                    rr_pair(ne, rd, ln, p, q);
                    const double app = G[p * K::LD + p], aqq = G[q * K::LD + q], apq = G[p * K::LD + q];
                    double cc = 1.0, ss = 0.0;
                    if (fabs(apq) > floor_abs && fabs(apq) > rel_tol * sqrt(fabs(app * aqq))) {
                        const double tau = (aqq - app) / (2.0 * apq);
                        const double t = copysign(1.0, tau) / (fabs(tau) + sqrt(1.0 + tau * tau));
                        cc = 1.0 / sqrt(1.0 + t * t);
                        ss = t * cc;
                        rotated = true;
                    }
                    pq[ln] = make_int2(p, q);
                    cs[ln] = make_double2(cc, ss);
                }
                __syncwarp();
                // columns p, q of G and V: lane = row
                for (int k = 0; k < half; ++k) {
                    const double2 r2 = cs[k];
                    if (r2.y == 0.0) continue;
                    const int2 k2 = pq[k];
                    double* gr = G + ln * K::LD;
                    double* vr = V + ln * K::LD;
                    const double gp = gr[k2.x], gq = gr[k2.y], vp = vr[k2.x], vq = vr[k2.y];
                    gr[k2.x] = r2.x * gp - r2.y * gq;
                    gr[k2.y] = r2.y * gp + r2.x * gq;
                    vr[k2.x] = r2.x * vp - r2.y * vq;
                    vr[k2.y] = r2.y * vp + r2.x * vq;
                }
                __syncwarp();
                // rows p, q of G: lane = column
                for (int k = 0; k < half; ++k) {
                    const double2 r2 = cs[k];
                    if (r2.y == 0.0) continue;
                    const int2 k2 = pq[k];
                    double* gp_ = G + k2.x * K::LD + ln;
                    double* gq_ = G + k2.y * K::LD + ln;
                    const double gp = *gp_, gq = *gq_;
                    *gp_ = r2.x * gp - r2.y * gq;
                    *gq_ = r2.y * gp + r2.x * gq;
                }
                __syncwarp();
            }
            if (!__any_sync(FULL, rotated)) break;
        }

        // ---- descending order, s, rank, Vt
        // NaN first, as in eig_sort_kernel and the reference's argsort()[::-1], so both svd_batched routes agree; sigma of a
        // NaN eigenvalue is NaN, not 0
        const double lam = ln >= n ? 0.0 : (nonfinite ? eig_nan() : scalbn(G[ln * K::LD + ln], e));
        int rk = 0;
        for (int j = 0; j < n; ++j) rk += eig_desc_before(__shfl_sync(FULL, lam, j), j, lam, ln);
        const double sv = sqrt_clip0(lam);
        if (ln < n) {
            src[rk] = ln;
            S[b * n + rk] = sv;
        }
        const unsigned above = __ballot_sync(FULL, ln < n && sv > tol);
        if (ln == 0) rank[b] = __popc(above);
        __syncwarp();
        if (ln < n)
            for (int r = 0; r < n; ++r) __stcs(Vt + (b * n + r) * n + ln, V[ln * K::LD + src[r]]);

        // ---- U = A (v_j / s_j) on the sorted columns: lane c owns column c (its V column and s come from lane src[c])
        const int from = ln < n ? src[ln] : 0;
        const double sc = __shfl_sync(FULL, sv, from);
        const bool keep = ln < n && sc > tol;
        double w[K::NMAX];
#pragma unroll
        for (int k = 0; k < K::NMAX; ++k) w[k] = (keep && k < n) ? V[k * K::LD + from] / sc : 0.0;
        __syncwarp();  // V's storage becomes the tile buffer again
        for (int r0 = 0; r0 < m; r0 += rows_per_tile) {
            const int rows = min(rows_per_tile, m - r0);
            load_tile(r0, rows);
            for (int r = 0; r < rows; ++r) {
                const double* row = stage + r * n;
                double acc = 0.0;
#pragma unroll
                for (int k = 0; k < K::NMAX; ++k)
                    if (k < n) acc = fma(row[k], w[k], acc);
                if (ln < n) __stcs(U + (b * m + r0 + r) * n + ln, keep ? acc : 0.0);
            }
            __syncwarp();
        }
    }
}

}  // namespace lq

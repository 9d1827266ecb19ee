// Streaming Householder R-factor kernel ("[R; block]" / TPQRT-style), one CTA per problem or per
// row range.  It is the engine of
//   K3  batched least squares  (linalg/qr.py:122-134): [A | B] streamed in 64-row blocks, R and
//       Q^T B kept in shared memory, back-substitution at the end -- Q is never formed;
//   K5a TSQR leaves / tree nodes: every CTA reduces its row range to one n x n R factor.
//
// Layout: lane l owns the folded column slots col(s, l) = 32 s + l (s even) or 32 (s+1) - 1 - l
// (s odd), warp w owns RPT consecutive rows of the current block, so a lane holds C x RPT doubles
// in registers.  Column step j of a block: the owning lane publishes its RPT entries of column j
// to a warp-private buffer, every lane forms x^T B[:, c] for its columns, the per-warp partials
// meet in shared memory (one __syncthreads per step, double buffered), and every warp redundantly
// builds  v = [R_jj + alpha ; x],  beta = 2 / v^T v  and updates its rows; warp 0 updates row j
// of R.  Starting from R = 0 makes the first block an ordinary Householder step.
#pragma once

#include "common.cuh"

namespace lq {

template <int C, int RPT, int WARPS>
struct StreamCfg {
    static constexpr int NCAP = 32 * C;          // column capacity
    static constexpr int BLOCK_ROWS = WARPS * RPT;
    static constexpr int RP = NCAP;              // pitch of R in shared memory
    __host__ __device__ static constexpr int col(int s, int l) { return (s & 1) ? (32 * (s + 1) - 1 - l) : (32 * s + l); }
    // shared doubles: R (nf x NCAP) + partials (2 x WARPS x NCAP) + vbuf (WARPS x RPT)
    __host__ static size_t smem_doubles(int nf) { return (size_t)nf * NCAP + 2 * WARPS * NCAP + WARPS * RPT + 8; }
};

// One block step-loop over the factored columns.  r: block registers; Rs: shared R.
// EXACT_ZERO_SKIP: skip a reflector only when the carried column [R_jj ; x] is exactly zero.  A block sees only part of the
// remaining column, so it cannot apply the reference's test (remaining norm < 1e-12, linalg/qr.py:79-80) to the whole
// column, and the rows of a skipped block would be dropped with the block: a column of norm 1.5e-12 spread over several
// blocks would end with R_jj = 0.  Without the skip, |R_jj| ends as the full remaining norm, on which the least-squares
// kernel's singularity report acts.
template <int C, int RPT, int WARPS, bool EXACT_ZERO_SKIP = false>
__device__ __forceinline__ void stream_factor_block(double (&r)[C][RPT], double* __restrict__ Rs, double* __restrict__ part,
                                                    double* __restrict__ vbuf, int nf, int lane, int warp) {
    using Cfg = StreamCfg<C, RPT, WARPS>;
    constexpr int NCAP = Cfg::NCAP;
    int colv[C];
#pragma unroll
    for (int s = 0; s < C; ++s) colv[s] = Cfg::col(s, lane);
    double* myv = vbuf + warp * RPT;

    for (int j = 0; j < nf; ++j) {
        const int so = j >> 5;
        const int lo = (so & 1) ? (32 * (so + 1) - 1 - j) : (j - 32 * so);
        const int par = j & 1;
        // owner lane publishes its rows of column j
        if (lane == lo) {
#pragma unroll
            for (int s = 0; s < C; ++s)
                if (s == so) {
#pragma unroll
                    for (int ii = 0; ii < RPT; ii += 2) *reinterpret_cast<double2*>(myv + ii) = make_double2(r[s][ii], r[s][ii + 1]);
                }
        }
        // old row j of R (read before the barrier, rewritten by warp 0 after it)
        double rrow[C];
#pragma unroll
        for (int s = 0; s < C; ++s) rrow[s] = Rs[j * NCAP + colv[s]];
        const double x0 = Rs[j * NCAP + j];
        __syncwarp();
        double xv[RPT];
#pragma unroll
        for (int ii = 0; ii < RPT; ii += 2) {
            const double2 t2 = *reinterpret_cast<const double2*>(myv + ii);
            xv[ii] = t2.x;
            xv[ii + 1] = t2.y;
        }
        double d[C];
#pragma unroll
        for (int s = 0; s < C; ++s) {
            double a0 = 0.0, a1 = 0.0;
            if (s >= so) {
#pragma unroll
                for (int ii = 0; ii < RPT; ii += 2) {
                    a0 = fma(xv[ii], r[s][ii], a0);
                    a1 = fma(xv[ii + 1], r[s][ii + 1], a1);
                }
            }
            d[s] = a0 + a1;
            part[(par * WARPS + warp) * NCAP + colv[s]] = d[s];
        }
        __syncthreads();
        double tot[C];
#pragma unroll
        for (int s = 0; s < C; ++s) {
            double t = 0.0;
#pragma unroll
            for (int ww = 0; ww < WARPS; ++ww) t += part[(par * WARPS + ww) * NCAP + colv[s]];
            tot[s] = t;
        }
        // sum of squares of the block part of column j lives in lane lo, slot so
        double ssb = 0.0;
#pragma unroll
        for (int s = 0; s < C; ++s)
            if (s == so) ssb = tot[s];
        ssb = __shfl_sync(0xffffffffu, ssb, lo);
        const double ss = fma(x0, x0, ssb);
        double rinv;
        const double nrm = sqrt_nr_t<2>(fmax(ss, 1e-300), rinv);
        const bool skip = EXACT_ZERO_SKIP ? (ss == 0.0) : (nrm < kEps);  // qr.py:79-80
        const double alpha = copysign(nrm, x0);
        const double v0 = x0 + alpha;
        const double beta = skip ? 0.0 : rcp_nr_t<2>(nrm * fabs(v0));
        double sc[C];
#pragma unroll
        for (int s = 0; s < C; ++s) {
            const double g = fma(v0, rrow[s], tot[s]);  // v^T [R_j,c ; B[:, c]]
            sc[s] = (colv[s] > j) ? beta * g : 0.0;
        }
#pragma unroll
        for (int s = 0; s < C; ++s) {
            if (s >= so) {
#pragma unroll
                for (int ii = 0; ii < RPT; ++ii) r[s][ii] = fma(-sc[s], xv[ii], r[s][ii]);
            }
        }
        if (warp == 0) {
#pragma unroll
            for (int s = 0; s < C; ++s) {
                const int c = colv[s];
                if (c > j) Rs[j * NCAP + c] = fma(-sc[s], v0, rrow[s]);
                else if (c == j && !skip) Rs[j * NCAP + c] = -alpha;
            }
        }
    }
    __syncthreads();
}

// ---------------------------------------------------------------------------------------------
// K3: batched Householder least squares, one CTA per system.  A (batch, m, n), B (batch, m, nrhs),
// X (batch, n, nrhs); n <= 64 (two column slots for A), nrhs <= 32 (third slot).  info (may be null): per system 0, or
// 1 + the first column whose R[j][j] is exactly 0 (np.linalg.solve raises there, linalg/qr.py:134).
// ---------------------------------------------------------------------------------------------
template <int RPT, int WARPS>
__global__ void __launch_bounds__(WARPS * 32)
    lstsq_stream_kernel(const double* __restrict__ A, const double* __restrict__ B, double* __restrict__ X,
                        int* __restrict__ info, int m, int n, int nrhs) {
    constexpr int C = 3;
    using Cfg = StreamCfg<C, RPT, WARPS>;
    constexpr int NCAP = Cfg::NCAP;
    extern __shared__ __align__(16) double sm[];
    double* Rs = sm;                                  // n x NCAP   (columns 64.. hold Q^T B)
    double* part = Rs + (size_t)n * NCAP;
    double* vbuf = part + 2 * WARPS * NCAP;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long sys = blockIdx.x;
    const double* Ag = A + sys * (long long)m * n;
    const double* Bg = B + sys * (long long)m * nrhs;

    for (int e = threadIdx.x; e < n * NCAP; e += WARPS * 32) Rs[e] = 0.0;
    __syncthreads();

    int colv[C];
#pragma unroll
    for (int s = 0; s < C; ++s) colv[s] = Cfg::col(s, lane);

    for (int rb = 0; rb < m; rb += Cfg::BLOCK_ROWS) {
        double r[C][RPT];
#pragma unroll
        for (int ii = 0; ii < RPT; ++ii) {
            const int row = rb + warp * RPT + ii;
            const bool ok = row < m;
#pragma unroll
            for (int s = 0; s < 2; ++s) r[s][ii] = (ok && colv[s] < n) ? ld_stream(Ag + (long long)row * n + colv[s]) : 0.0;
            const int cb = colv[2] - 64;
            r[2][ii] = (ok && cb < nrhs) ? ld_stream(Bg + (long long)row * nrhs + cb) : 0.0;
        }
        stream_factor_block<C, RPT, WARPS, true>(r, Rs, part, vbuf, n, lane, warp);
    }

    if (info != nullptr && threadIdx.x == 0) {
        int bad = 0;
        for (int j = n - 1; j >= 0; --j)
            if (Rs[j * NCAP + j] == 0.0) bad = j + 1;
        info[sys] = bad;
    }
    // back-substitution R x = y, y = Rs[:, 64 + k]; one thread per right-hand side
    if (threadIdx.x < nrhs) {
        const int k = 64 + threadIdx.x;
        for (int i = n - 1; i >= 0; --i) {
            double acc = Rs[i * NCAP + k];
            for (int c = i + 1; c < n; ++c) acc = fma(-Rs[i * NCAP + c], Rs[c * NCAP + k], acc);
            Rs[i * NCAP + k] = acc / Rs[i * NCAP + i];
        }
    }
    __syncthreads();
    double* Xg = X + sys * (long long)n * nrhs;
    for (int e = threadIdx.x; e < n * nrhs; e += WARPS * 32) {
        const int i = e / nrhs, k = e - i * nrhs;
        Xg[e] = Rs[i * NCAP + 64 + k];
    }
}

// ---------------------------------------------------------------------------------------------
// K5a: R factor of a row range of a tall-skinny matrix (n <= 128).  CTA b reduces rows
// [b * rows_per_cta, ...) of A (m x n, lda) to an upper-triangular n x n factor Rout[b].
// ---------------------------------------------------------------------------------------------
template <int RPT, int WARPS>
__global__ void __launch_bounds__(WARPS * 32)
    tsqr_leaf_kernel(const double* __restrict__ A, int lda, long long m, int n, long long rows_per_cta,
                     double* __restrict__ Rout) {
    constexpr int C = 4;
    using Cfg = StreamCfg<C, RPT, WARPS>;
    constexpr int NCAP = Cfg::NCAP;
    extern __shared__ __align__(16) double sm[];
    double* Rs = sm;
    double* part = Rs + (size_t)n * NCAP;
    double* vbuf = part + 2 * WARPS * NCAP;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long row0 = blockIdx.x * rows_per_cta;
    const long long row1 = min(m, row0 + rows_per_cta);

    for (int e = threadIdx.x; e < n * NCAP; e += WARPS * 32) Rs[e] = 0.0;
    __syncthreads();
    int colv[C];
#pragma unroll
    for (int s = 0; s < C; ++s) colv[s] = Cfg::col(s, lane);

    for (long long rb = row0; rb < row1; rb += Cfg::BLOCK_ROWS) {
        double r[C][RPT];
#pragma unroll
        for (int ii = 0; ii < RPT; ++ii) {
            const long long row = rb + warp * RPT + ii;
            const bool ok = row < row1;
#pragma unroll
            for (int s = 0; s < C; ++s) r[s][ii] = (ok && colv[s] < n) ? ld_stream(A + row * lda + colv[s]) : 0.0;
        }
        stream_factor_block<C, RPT, WARPS>(r, Rs, part, vbuf, n, lane, warp);
    }
    double* Rg = Rout + (long long)blockIdx.x * n * n;
    for (int e = threadIdx.x; e < n * n; e += WARPS * 32) {
        const int i = e / n, c = e - i * n;
        Rg[e] = (c >= i) ? Rs[i * NCAP + c] : 0.0;
    }
}

}  // namespace lq

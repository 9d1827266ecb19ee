// TSQR (SURVEY.md section 8 row a7) and least squares on its pipeline: the Householder reduction tree of R factors,
// CholeskyQR2 for n <= 128, block Gram-Schmidt over CholeskyQR2 panels for n > 128, the blocked Householder fallbacks, and
// the NCCL exchange steps of the row-sharded variants.
#include <algorithm>
#include <vector>

#include "../../include/linalg_b200.h"
#include "ops.cuh"
#include "stream_qr.cuh"

namespace lq {

namespace {

// ------------------------------------------------------------------ small triangular helpers (single CTA)
// make diag(R) > 0: R <- S R, and return S (n) so that Q <- Q S
__global__ void __launch_bounds__(256) sign_fix_R_kernel(double* __restrict__ R, int n, double* __restrict__ sgn) {
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const double sg = (R[(size_t)i * n + i] < 0.0) ? -1.0 : 1.0;
        sgn[i] = sg;
    }
    __syncthreads();
    for (int e = threadIdx.x; e < n * n; e += blockDim.x) {
        const int i = e / n;
        R[e] *= sgn[i];
    }
}

// ---- register-resident kernels for n <= 128.  Every caller has n <= 128: tsqr_local sends wider matrices to tsqr_wide,
// whose panels are at most 128 columns.  The CholeskyQR2 path of TSQR runs two of each per call; shared-memory
// versions cost 0.20 + 0.36 ms, a fifth of the whole 2^20 x 128 TSQR.
//
// Inverse of an upper-triangular R: warp w solves the columns w, w + 32, w + 64, w + 96 of R X = I together (four
// independent recurrences interleaved); lane l holds rows l + 32 u of each right-hand side in registers, R sits in
// shared memory (odd pitch: a column walk is conflict free), 1 / R_kk is formed once.  Column-oriented back
// substitution: x_k is broadcast from its owner lane, every lane updates its rows above k.
// The 32 warps (4 columns each) are independent: they run as 8 CTAs of 4 warps on 8 SMs (one CTA of 32 warps was bound by
// the issue rate of a single SM: 45 us; every CTA stages its own copy of R from L2).
__global__ void __launch_bounds__(128) triu_inverse128_kernel(const double* __restrict__ R, int n, double* __restrict__ Rinv) {
    extern __shared__ double ti_sm[];
    double (*S)[129] = reinterpret_cast<double (*)[129]>(ti_sm);
    __shared__ double dinv[128];
    const int tid = threadIdx.x, w = blockIdx.x * (blockDim.x >> 5) + (tid >> 5), ln = tid & 31;
    for (int e = tid; e < 128 * 128; e += blockDim.x) {
        const int i = e >> 7, k = e & 127;
        S[i][k] = (i < n && k < n) ? R[(size_t)i * n + k] : ((i == k) ? 1.0 : 0.0);
    }
    __syncthreads();
    if (tid < 128) dinv[tid] = 1.0 / S[tid][tid];
    __syncthreads();
    double x[4][4];  // [column c = w + 32 cc][row block u]: row ln + 32 u
#pragma unroll
    for (int cc = 0; cc < 4; ++cc)
#pragma unroll
        for (int u = 0; u < 4; ++u) x[cc][u] = (ln + 32 * u == w + 32 * cc) ? 1.0 : 0.0;
#pragma unroll
    for (int ub = 3; ub >= 0; --ub) {
        for (int kk = 31; kk >= 0; --kk) {
            const int k = 32 * ub + kk;
            const double dk = dinv[k];
            double rk[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) rk[u] = (u <= ub) ? S[ln + 32 * u][k] : 0.0;
#pragma unroll
            for (int cc = 0; cc < 4; ++cc) {
                if (cc < ub) continue;  // column w + 32 cc < 32 (cc + 1) <= k: x_k = 0 (compile-time skip of whole blocks)
                const double xk = __shfl_sync(0xffffffffu, x[cc][ub], kk) * dk;
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    if (u < ub) x[cc][u] = fma(-rk[u], xk, x[cc][u]);
                    else if (u == ub) x[cc][u] = (ln == kk) ? xk : ((ln < kk) ? fma(-rk[u], xk, x[cc][u]) : x[cc][u]);
                }
            }
        }
    }
#pragma unroll
    for (int cc = 0; cc < 4; ++cc) {
        const int col = w + 32 * cc;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = ln + 32 * u;
            if (i < n && col < n) Rinv[(size_t)i * n + col] = (i <= col) ? x[cc][u] : 0.0;
        }
    }
}

// Upper Cholesky factor for n <= 128 with the matrix in registers: thread (ty, tx) of a 32 x 32 block owns the
// elements (ty + 32 a, tx + 32 b).  Per column: the diagonal owner publishes the pivot, the owners of row j publish
// the scaled row, everybody updates its 16 elements (8 shared loads, 16 FMAs, no index arithmetic).
// stat[0] = 1 if a pivot is not safely positive (breakdown), stat[1] = max_j G_jj / min_j R_jj^2  (~ cond(A)^2).
__global__ void __launch_bounds__(1024) chol_upper128_kernel(const double* __restrict__ G, int n, double* __restrict__ R,
                                                             double* __restrict__ stat) {
    __shared__ double rowbuf[2][128];
    __shared__ double s_piv[2];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    double a[4][4];
#pragma unroll
    for (int ia = 0; ia < 4; ++ia)
#pragma unroll
        for (int ib = 0; ib < 4; ++ib) {
            const int i = ty + 32 * ia, k = tx + 32 * ib;
            a[ia][ib] = (i < n && k < n) ? G[(size_t)i * n + k] : ((i == k) ? 1.0 : 0.0);
        }
    double dmax = 0.0, pmin = 1e300;
    if (threadIdx.x == 0) {
        for (int j = 0; j < n; ++j) dmax = fmax(dmax, G[(size_t)j * n + j]);
    }
    int bad = 0;
#pragma unroll
    for (int ja = 0; ja < 4; ++ja) {
        for (int jj = 0; jj < 32; ++jj) {
            const int j = 32 * ja + jj, par = j & 1;
            if (ty == jj && tx == jj) s_piv[par] = a[ja][ja];
            __syncthreads();
            const double piv = s_piv[par];
            if (!(piv > 0.0)) {  // also catches NaN; uniform
                bad = 1;
                break;
            }
            if (j < n) pmin = fmin(pmin, piv);  // (rows >= n are identity padding)
            const double rd = rsqrt_nr_t<2>(piv);
            if (ty == jj) {
                // my elements of row j, scaled; columns left of the diagonal are not part of R
#pragma unroll
                for (int ib = 0; ib < 4; ++ib) {
                    const int k = tx + 32 * ib;
                    double v = a[ja][ib] * rd;
                    if (k == j) v = piv * rd;
                    if (k < j) v = 0.0;
                    a[ja][ib] = v;
                    rowbuf[par][k] = v;
                }
            }
            __syncthreads();
            double ri[4], rk[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                ri[q] = rowbuf[par][ty + 32 * q];
                rk[q] = rowbuf[par][tx + 32 * q];
            }
#pragma unroll
            for (int ia = 0; ia < 4; ++ia) {
                if (ia < ja) continue;
                const int i = ty + 32 * ia;
#pragma unroll
                for (int ib = 0; ib < 4; ++ib) {
                    if (ib < ja) continue;
                    if (i > j) a[ia][ib] = fma(-ri[ia], rk[ib], a[ia][ib]);  // rows below j (columns left of j see rk = 0)
                }
            }
        }
        if (bad) break;
    }
#pragma unroll
    for (int ia = 0; ia < 4; ++ia)
#pragma unroll
        for (int ib = 0; ib < 4; ++ib) {
            const int i = ty + 32 * ia, k = tx + 32 * ib;
            if (i < n && k < n) R[(size_t)i * n + k] = (k >= i) ? a[ia][ib] : 0.0;
        }
    if (threadIdx.x == 0) {
        stat[0] = bad ? 1.0 : 0.0;
        stat[1] = bad ? 1e300 : dmax / pmin;
    }
}

int launch_triu_inverse(Ctx* c, const double* R, int n, double* Rinv) {
    LQ_REQUIRE(c, n <= 128, LQ_ERR_UNSUPPORTED, "triangular inverse supports n <= 128 (got %d)", n);
    return launch<triu_inverse128_kernel>(c, 8, 128, 128 * 129 * 8, c->stream, 128 * 129 * 8, R, n, Rinv);
}

// M <- M diag(sgn)   (rows x n)
__global__ void __launch_bounds__(256) scale_cols_tall_kernel(double* __restrict__ M, long long rows, int n,
                                                              const double* __restrict__ sgn) {
    const long long total = rows * n;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x)
        M[e] *= sgn[e % n];
}

// R factor (n x n upper) of A (m x n, lda) by a tree of streaming Householder reductions
int tsqr_rfactor(Ctx* c, const double* A, int lda, long long m, int n, double* R /* n x n */) {
    using Cfg = StreamCfg<4, 16, 8>;
    const size_t smem = Cfg::smem_doubles(n) * sizeof(double);
    const double* cur = A;
    int cur_ld = lda;
    long long cur_m = m;
    DevBuf bufs[2];
    int flip = 0;
    for (int level = 0; level < 8; ++level) {
        // leaves of >= 4 blocks each, at most 2 CTAs per SM worth of leaves
        long long min_rows = (long long)Cfg::BLOCK_ROWS * 8;
        long long ctas = std::max<long long>(1, std::min<long long>((long long)c->sm_count, cur_m / min_rows));
        if (level > 0) ctas = std::max<long long>(1, std::min<long long>(ctas, cur_m / ((long long)n * 8)));
        long long rpc = (cur_m + ctas - 1) / ctas;
        rpc = (rpc + Cfg::BLOCK_ROWS - 1) / Cfg::BLOCK_ROWS * Cfg::BLOCK_ROWS;
        ctas = (cur_m + rpc - 1) / rpc;
        double* out;
        if (ctas == 1) {
            out = R;
        } else {
            LQ_TRY(bufs[flip].alloc(c, sizeof(double) * (size_t)ctas * n * n));
            out = bufs[flip].as<double>();
        }
        LQ_TRY((launch<tsqr_leaf_kernel<16, 8>>(c, (unsigned)ctas, 256, smem, c->stream, SMEM_OPT_IN_REST, cur, cur_ld, cur_m, n,
                                                rpc, out)));
        if (ctas == 1) return LQ_OK;
        cur = out;
        cur_ld = n;
        cur_m = ctas * (long long)n;
        flip ^= 1;
    }
    set_error(c, "tsqr_rfactor: reduction tree did not terminate");
    return LQ_ERR_ARG;
}

}  // namespace

// R factor of a row-sharded A (local block m x n, row stride lda): the reduction tree of the local block, then the tree of
// the all-gathered stack of local factors (Rall: nranks x n x n), so that every rank ends with the same R
static int sharded_rfactor(Ctx* c, const double* A, int lda, long long m, int n, double* Rall, double* R) {
    LQ_TRY(tsqr_rfactor(c, A, lda, m, n, R));
    LQ_TRY(comm_allgather(c, R, Rall, (long long)n * n));
    return tsqr_rfactor(c, Rall, n, (long long)c->nranks * n, n, R);
}

// robust path of one GPU for ill-conditioned (or nearly square) input: the blocked compact-WY Householder QR, whose Q is
// formed from the reflectors (residual and orthogonality O(eps) for any cond(A)), flipped to diag(R) > 0
static int tsqr_blocked_fallback(Ctx* c, const double* A, long long m, int n, double* Q, double* R) {
    DevBuf sgn;
    LQ_TRY(sgn.alloc(c, sizeof(double) * n));
    LQ_TRY(blocked_householder_qr(c, A, (int)m, n, Q, R));
    LQ_TRY(launch<sign_fix_R_kernel>(c, 1, 256, 0, c->stream, 0, R, n, sgn.as<double>()));
    return launch<scale_cols_tall_kernel>(c, grid_for(c, m * n), 256, 0, c->stream, 0, Q, m, n, sgn.as<double>());
}

// TSQR of a row-sharded A: R by the Householder reduction tree (leaves stream their rows, R factors are combined),
// Q = A R^{-1} followed by one TSQR refinement pass (restores orthogonality to O(eps) whenever
// cond(A) * eps << 1), signs normalised so that diag(R) > 0 -- the MGS convention (qr.py:39-42).
static int tsqr_householder(Ctx* c, const double* A, long long m, int n, double* Q, double* R) {
    DevBuf R1, R2, Rinv, Rall, sgn, Q1;
    const size_t nn = sizeof(double) * (size_t)n * n;
    LQ_TRY(R1.alloc(c, nn));
    LQ_TRY(R2.alloc(c, nn));
    LQ_TRY(Rinv.alloc(c, nn));
    LQ_TRY(sgn.alloc(c, sizeof(double) * n));
    LQ_TRY(Q1.alloc(c, sizeof(double) * (size_t)m * n));
    LQ_TRY(Rall.alloc(c, nn * c->nranks));
    // pass 1
    LQ_TRY(sharded_rfactor(c, A, n, m, n, Rall.as<double>(), R1.as<double>()));
    LQ_TRY(launch_triu_inverse(c, R1.as<double>(), n, Rinv.as<double>()));
    LQ_TRY(gemm(c, false, false, m, n, n, 1.0, A, n, Rinv.as<double>(), n, 0.0, Q1.as<double>(), n));
    // pass 2 (refinement)
    LQ_TRY(sharded_rfactor(c, Q1.as<double>(), n, m, n, Rall.as<double>(), R2.as<double>()));
    LQ_TRY(launch<sign_fix_R_kernel>(c, 1, 256, 0, c->stream, 0, R2.as<double>(), n, sgn.as<double>()));  // R2 <- S R2 (temporarily, S folded below)
    // we want R = S' (R2 R1) with diag > 0.  Compute R = R2 R1 first with the unsigned R2:
    //   sign_fix made diag(R2) > 0; R1's diagonal sign decides the final flip.
    LQ_TRY(gemm(c, false, false, n, n, n, 1.0, R2.as<double>(), n, R1.as<double>(), n, 0.0, R, n));
    // Q = Q1 (S R2)^{-1} ... then flip so that diag(R) > 0
    LQ_TRY(launch_triu_inverse(c, R2.as<double>(), n, Rinv.as<double>()));
    LQ_TRY(launch<sign_fix_R_kernel>(c, 1, 256, 0, c->stream, 0, R, n, sgn.as<double>()));  // R <- S2 R
    LQ_TRY(launch<scale_cols_tall_kernel>(c, grid_for(c, (long long)n * n), 256, 0, c->stream, 0, Rinv.as<double>(), (long long)n,
                                          n, sgn.as<double>()));  // Rinv <- Rinv S2
    LQ_TRY(gemm(c, false, false, m, n, n, 1.0, Q1.as<double>(), n, Rinv.as<double>(), n, 0.0, Q, n));
    return LQ_OK;
}

// Fast path for well-conditioned tall-skinny matrices: CholeskyQR2 on the FP64 tensor pipe.
//   G1 = A^T A (+ all-reduce over the row shards) -> R1 = chol(G1) -> Q1 = A R1^{-1}
//   G2 = Q1^T Q1 (+ all-reduce)                   -> R2 = chol(G2) -> Q  = Q1 R2^{-1},  R = R2 R1
// Four streaming GEMMs instead of two column-by-column Householder sweeps; diag(R) > 0 by construction (the
// convention of linalg/qr.py:39-42).  The second pass restores orthogonality to O(eps) as long as
// cond(A)^2 * eps << 1; the Cholesky kernel reports a cond(A)^2 estimate and the Householder TSQR tree below
// takes over when it exceeds 1e10 (or a pivot breaks down).
__global__ void tsqr_flags_kernel(double* f, double a, double b) {
    f[0] = a;
    f[1] = b;
}

// status words of one CholeskyQR2 (stat[0..3] of cholqr2_enqueue), identical on every rank (they derive from all-reduced data)
struct CholQrStatus {
    double chol1_bad = 0, cond2 = 0, chol2_bad = 0, cond2_pass2 = 0;
    double ranks_short = 0;  // number of ranks whose local block has fewer rows than columns
    CholQrStatus() = default;
    CholQrStatus(const double* stat, double short_count)
        : chol1_bad(stat[0]), cond2(stat[1] == stat[1] ? stat[1] : 1e300 /* NaN -> ill-conditioned */), chol2_bad(stat[2]),
          cond2_pass2(stat[3]), ranks_short(short_count) {}
    bool ok() const { return chol1_bad == 0.0 && cond2 < 1e10 && chol2_bad == 0.0; }
};

// scratch of the CholeskyQR2 pipeline (allocated once per call, reused by every column panel of tsqr_wide); nrhs > 0 adds
// what least squares needs besides: [G2 | C], R2^-1 and the two n x nrhs intermediates of its tail
struct CholQrScratch {
    DevBuf G, R1, R2, Rinv, Q1;
    DevBuf GC, R2inv, Y, Z;
    int alloc(Ctx* c, long long m, int n, int nrhs = 0) {
        const size_t nn = sizeof(double) * (size_t)n * n, nk = sizeof(double) * (size_t)n * nrhs;
        LQ_TRY(G.alloc(c, nn + 2 * sizeof(double)));
        LQ_TRY(R1.alloc(c, nn));
        LQ_TRY(R2.alloc(c, nn));
        LQ_TRY(Rinv.alloc(c, nn));
        LQ_TRY(Q1.alloc(c, sizeof(double) * (size_t)m * n));
        if (nrhs > 0) {
            LQ_TRY(GC.alloc(c, nn + nk));
            LQ_TRY(R2inv.alloc(c, nn));
            LQ_TRY(Y.alloc(c, nk));
            LQ_TRY(Z.alloc(c, nk));
        }
        return LQ_OK;
    }
};

// Pass 1 of CholeskyQR2 of the m x n block A (row stride lda, n <= 128), into w: G = A^T A (+ all-reduce over the row shards)
// -> R1 = chol(G) -> Rinv = R1^-1 -> Q1 = A Rinv.  stat[0..1] (device) receive chol1_bad and the cond^2 estimate.
// `short_flag` >= 0 puts that value into the two spare words behind G so that it is summed over the ranks by the all-reduce
// (G[n*n]).
static int cholqr_pass(Ctx* c, const double* A, int lda, long long m, int n, bool sharded, double short_flag, CholQrScratch& w,
                       double* stat) {
    double* G = w.G.as<double>();
    const bool carry = short_flag >= 0.0;
    if (carry) LQ_TRY(launch<tsqr_flags_kernel>(c, 1, 1, 0, c->stream, 0, G + (size_t)n * n, short_flag, 0.0));
    LQ_TRY(gram(c, A, lda, m, n, G));
    if (sharded) LQ_TRY(comm_allreduce_sum(c, G, (long long)n * n + (carry ? 2 : 0)));
    LQ_TRY(launch<chol_upper128_kernel>(c, 1, 1024, 0, c->stream, 0, G, n, w.R1.as<double>(), stat));
    LQ_TRY(launch_triu_inverse(c, w.R1.as<double>(), n, w.Rinv.as<double>()));
    return gemm(c, false, false, m, n, n, 1.0, A, lda, w.Rinv.as<double>(), n, 0.0, w.Q1.as<double>(), n);
}

// Enqueue one CholeskyQR2 of the m x n block A (row stride lda, n <= 128) -> Q (ldq), R (ldr); nothing is read back.
// stat[0..3] (device) receive chol1_bad, cond^2 estimate, chol2_bad, cond^2 of pass 2; short_flag as in cholqr_pass.
static int cholqr2_enqueue(Ctx* c, const double* A, int lda, long long m, int n, double* Q, int ldq, double* R, int ldr,
                           bool sharded, CholQrScratch& w, double* stat, double short_flag) {
    double* G = w.G.as<double>();
    LQ_TRY(cholqr_pass(c, A, lda, m, n, sharded, short_flag, w, stat));
    // pass 2
    LQ_TRY(gram(c, w.Q1.as<double>(), n, m, n, G));
    if (sharded) LQ_TRY(comm_allreduce_sum(c, G, (long long)n * n));
    LQ_TRY(launch<chol_upper128_kernel>(c, 1, 1024, 0, c->stream, 0, G, n, w.R2.as<double>(), stat + 2));
    LQ_TRY(launch_triu_inverse(c, w.R2.as<double>(), n, w.Rinv.as<double>()));
    LQ_TRY(gemm(c, false, false, n, n, n, 1.0, w.R2.as<double>(), n, w.R1.as<double>(), n, 0.0, R, ldr));
    LQ_TRY(gemm(c, false, false, m, n, n, 1.0, w.Q1.as<double>(), n, w.Rinv.as<double>(), n, 0.0, Q, ldq));
    return LQ_OK;
}

// the one read-back of a CholeskyQR2 call, behind everything else on the stream: stat[0..3] and the short-rank count that
// the first all-reduce summed behind G
static int read_cholqr_status(Ctx* c, const double* stat, const CholQrScratch& w, int n, CholQrStatus* st) {
    double h[6] = {0, 0, 0, 0, 0, 0};
    LQ_CUDA(c, cudaMemcpyAsync(h, stat, 4 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    LQ_CUDA(c, cudaMemcpyAsync(h + 4, w.G.as<double>() + (size_t)n * n, 2 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    LQ_CUDA(c, cudaStreamSynchronize(c->stream));
    *st = CholQrStatus(h, h[4]);
    return LQ_OK;
}

static int tsqr_cholqr2(Ctx* c, const double* A, long long m, int n, double* Q, double* R, bool sharded, CholQrStatus* st) {
    // Optimistic pipeline: nothing is read back until the last kernel is queued (round 1 synchronised with the host after
    // the first Cholesky to look at the cond^2 estimate: a bubble in the middle of a 4 ms call).  The status words and the
    // "short rank" count ride in the first all-reduce / are computed from all-reduced data, so every rank reaches the same
    // verdict and a fallback is taken by all ranks together (ADVICE r1: the path decision must be collective).
    CholQrScratch w;
    DevBuf stat;
    LQ_TRY(w.alloc(c, m, n));
    LQ_TRY(stat.alloc(c, 4 * sizeof(double)));
    LQ_TRY(cholqr2_enqueue(c, A, n, m, n, Q, n, R, n, sharded, w, stat.as<double>(), m < n ? 1.0 : 0.0));
    return read_cholqr_status(c, stat.as<double>(), w, n, st);
}

// *count = the number of ranks that pass flag = 1 (too few local rows for the reflector tree), summed over the ranks so that
// every rank reaches the same verdict
static int count_short_ranks(Ctx* c, double flag, double* count) {
    DevBuf f;
    LQ_TRY(f.alloc(c, 2 * sizeof(double)));
    LQ_TRY(launch<tsqr_flags_kernel>(c, 1, 1, 0, c->stream, 0, f.as<double>(), flag, 0.0));
    LQ_TRY(comm_allreduce_sum(c, f.as<double>(), 2));
    double h[2] = {0, 0};
    LQ_CUDA(c, cudaMemcpyAsync(h, f.p, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
    LQ_CUDA(c, cudaStreamSynchronize(c->stream));
    *count = h[0];
    return LQ_OK;
}

__global__ void add_inplace_kernel(double* __restrict__ dst, int ldd, const double* __restrict__ src, int lds, int rows, int cols) {
    const long long total = (long long)rows * cols;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const int i = (int)(e / cols), k = (int)(e % cols);
        dst[(size_t)i * ldd + k] += src[(size_t)i * lds + k];
    }
}

// a7 for n > 128 (e.g. the reference's own benchmark shape 5000 x 1000, linalg/benchmark_qr.py:17): block classical
// Gram-Schmidt with re-orthogonalisation (BCGS2) over 128-column panels, each panel factored by CholeskyQR2 --
//   W  = A_k - Q_prev S1,  S1 = Q_prev^T A_k        (first projection)
//   W' = W   - Q_prev S2,  S2 = Q_prev^T W          (second projection: orthogonality to O(eps))
//   W' = Q_k R_kk (CholeskyQR2, diag > 0)           R[prev, k] = S1 + S2
// everything is GEMMs on the FP64 tensor pipe; row-sharded calls all-reduce S1, S2 and the panel Gram matrices.  The
// status words of all panels are read back once at the end; any ill-conditioned panel sends the whole call to the
// reflector path (single GPU) or fails alike on every rank (sharded).
static int tsqr_wide(Ctx* c, const double* A, long long m, int n, double* Q, double* R, bool sharded) {
    const bool sh = sharded && c->nranks > 1;
    constexpr int PB = 128;
    const int np = (n + PB - 1) / PB;
    bool ok = !c->env_tsqr_householder && (sh || m >= 2LL * n);
    if (ok) {
        CholQrScratch w;
        DevBuf stat, S;
        LQ_TRY(w.alloc(c, m, PB));
        LQ_TRY(stat.alloc(c, sizeof(double) * 4 * np));
        LQ_TRY(S.alloc(c, sizeof(double) * (size_t)n * PB));
        LQ_CUDA(c, cudaMemsetAsync(R, 0, sizeof(double) * (size_t)n * n, c->stream));
        LQ_CUDA(c, cudaMemcpyAsync(Q, A, sizeof(double) * (size_t)m * n, cudaMemcpyDeviceToDevice, c->stream));
        for (int k = 0; k < np; ++k) {
            const int c0 = k * PB, bk = std::min(PB, n - c0);
            double* Qk = Q + c0;
            for (int pass = 0; pass < 2 && c0 > 0; ++pass) {
                LQ_TRY(gemm(c, true, false, c0, bk, (int)m, 1.0, Q, n, Qk, n, 0.0, S.as<double>(), bk));
                if (sh) LQ_TRY(comm_allreduce_sum(c, S.as<double>(), (long long)c0 * bk));
                LQ_TRY(gemm(c, false, false, m, bk, c0, -1.0, Q, n, S.as<double>(), bk, 1.0, Qk, n));
                LQ_TRY(launch<add_inplace_kernel>(c, grid_for(c, (long long)c0 * bk), 256, 0, c->stream, 0, R + c0, n, S.as<double>(),
                                                  bk, c0, bk));
            }
            LQ_TRY(cholqr2_enqueue(c, Qk, n, m, bk, Qk, n, R + (size_t)c0 * n + c0, n, sh, w, stat.as<double>() + 4 * k, -1.0));
        }
        std::vector<double> h(4 * (size_t)np);
        LQ_CUDA(c, cudaMemcpyAsync(h.data(), stat.p, sizeof(double) * h.size(), cudaMemcpyDeviceToHost, c->stream));
        LQ_CUDA(c, cudaStreamSynchronize(c->stream));
        for (int k = 0; k < np; ++k)
            if (!CholQrStatus(&h[4 * k], 0.0).ok()) ok = false;
        if (ok) return LQ_OK;
    }
    LQ_REQUIRE(c, !sh, LQ_ERR_UNSUPPORTED,
               "tsqr (sharded, n = %d > 128): a column panel is too ill-conditioned for CholeskyQR2 and the reflector tree "
               "supports n <= 128", n);
    LQ_REQUIRE(c, m >= n, LQ_ERR_SHAPE, "tsqr needs m >= n (got %lld x %d)", m, n);
    return tsqr_blocked_fallback(c, A, m, n, Q, R);
}

// a7: thin QR of a tall-skinny matrix with diag(R) > 0.
int tsqr_local(Ctx* c, const double* A, long long m, int n, double* Q, double* R, bool sharded) {
    const bool sh = sharded && c->nranks > 1;
    // Row-sharded calls validate only what every rank sees alike (n); the rank-local row count is checked through the
    // all-reduced "short rank" count so that no rank leaves while its peers wait in a collective.
    LQ_REQUIRE(c, n >= 1 && m >= 1 && (sh || m >= n), LQ_ERR_SHAPE, "tsqr needs m >= n >= 1 (got %lld x %d)", m, n);
    LQ_REQUIRE(c, m < (1LL << 31), LQ_ERR_SHAPE, "tsqr: more than 2^31 rows per device not supported");
    if (n > 128) return tsqr_wide(c, A, m, n, Q, R, sharded);
    CholQrStatus st;
    bool have_status = false;
    if (!c->env_tsqr_householder && (sh || m >= 4LL * n)) {
        LQ_TRY(tsqr_cholqr2(c, A, m, n, Q, R, sh, &st));
        if (st.ok()) return LQ_OK;
        have_status = true;
    }
    if (!sh) return tsqr_blocked_fallback(c, A, m, n, Q, R);
    // row-sharded and ill-conditioned: Householder reduction tree + Q = A R^{-1} with one refinement pass
    // (orthogonality O(eps), residual O(cond(A) eps)); its leaves need at least n rows on every rank
    if (!have_status) LQ_TRY(count_short_ranks(c, m < n ? 1.0 : 0.0, &st.ranks_short));
    LQ_REQUIRE(c, st.ranks_short == 0.0, LQ_ERR_SHAPE,
               "tsqr (sharded, reflector path): %d rank(s) hold fewer than n = %d rows; re-shard the rows", (int)st.ranks_short, n);
    return tsqr_householder(c, A, m, n, Q, R);
}

// ------------------------------------------------------------------ least squares on the tall-skinny pipeline
// X (n x nrhs) = R^-1 y from the top n rows [R | y] (pitch ld) of the R factor of [A | B]; info = 0, or 1 + the first j with
// R[j][j] exactly 0 (X is then not meaningful)
__global__ void __launch_bounds__(128) backsub_aug_kernel(const double* __restrict__ Rf, int ld, int n, int nrhs,
                                                          double* __restrict__ X, int* __restrict__ info) {
    if (threadIdx.x == 0) {
        int bad = 0;
        for (int j = 0; j < n && !bad; ++j)
            if (Rf[(size_t)j * ld + j] == 0.0) bad = j + 1;
        *info = bad;
    }
    for (int k = threadIdx.x; k < nrhs; k += blockDim.x)
        for (int i = n - 1; i >= 0; --i) {
            double s = Rf[(size_t)i * ld + n + k];
            for (int j = i + 1; j < n; ++j) s = fma(-Rf[(size_t)i * ld + j], X[(size_t)j * nrhs + k], s);
            X[(size_t)i * nrhs + k] = s / Rf[(size_t)i * ld + i];
        }
}

// [G | C] = Q^T [Q | B] (G n x n, C n x nrhs): the strip kernel where its shape rules allow it (an odd nrhs < 32 is padded with a
// zero column first, to the even width of the strip kernel's bulk copies), the SYRK or GEMM Gram matrix and a TN GEMM otherwise
static int gram_rhs(Ctx* c, const double* Q, long long m, int n, const double* B, int nrhs, double* G, double* C) {
    // (Q stands in for the padded copy of B in the check: both are 16-byte aligned workspace)
    if (nrhs % 2 == 1 && syrk_strip_supported(Q, m, n, Q, nrhs + 1)) {
        const int kp = nrhs + 1;
        DevBuf Bp, Cp;
        LQ_TRY(Bp.alloc(c, sizeof(double) * (size_t)m * kp));
        LQ_TRY(Cp.alloc(c, sizeof(double) * (size_t)n * kp));
        LQ_TRY(pad_columns(c, B, nrhs, Bp.as<double>(), kp, m, nrhs, kp));
        LQ_TRY(syrk_strip_tn(c, Q, m, n, Bp.as<double>(), kp, G, Cp.as<double>()));
        LQ_CUDA(c, cudaMemcpy2DAsync(C, sizeof(double) * nrhs, Cp.p, sizeof(double) * kp, sizeof(double) * nrhs, (size_t)n,
                                     cudaMemcpyDeviceToDevice, c->stream));
        return LQ_OK;
    }
    const int rc = syrk_strip_tn(c, Q, m, n, B, nrhs, G, C);
    if (rc != LQ_ERR_UNSUPPORTED) return rc;
    LQ_TRY(gram(c, Q, n, m, n, G));
    return gemm(c, true, false, n, nrhs, (int)m, 1.0, Q, n, B, nrhs, 0.0, C, nrhs);
}

// CholeskyQR2 least squares (n <= 128), never forming Q:
//   G1 = A^T A (+ all-reduce) -> R1 = chol(G1) -> Q1 = A R1^-1
//   [G2 | C] = Q1^T [Q1 | B] (+ one all-reduce of the packed buffer) -> R2 = chol(G2)
//   X = (R2 R1)^-1 R2^-T C = R1^-1 R2^-1 R2^-T C
// Everything is queued before the one read-back of the status words (cholqr2_enqueue's verdict).  CholeskyQR2 of [A | B] would
// break down for every consistent system (zero residual: [A | B] is rank deficient), so B only enters the second pass.
static int lstsq_cholqr2(Ctx* c, const double* A, long long m, int n, const double* B, int nrhs, double* X, bool sh,
                         double short_flag, CholQrStatus* st) {
    CholQrScratch w;
    DevBuf stat;
    LQ_TRY(w.alloc(c, m, n, nrhs));
    LQ_TRY(stat.alloc(c, 4 * sizeof(double)));
    double* G2 = w.GC.as<double>();
    double* C = G2 + (size_t)n * n;
    LQ_TRY(cholqr_pass(c, A, n, m, n, sh, short_flag, w, stat.as<double>()));
    // pass 2
    LQ_TRY(gram_rhs(c, w.Q1.as<double>(), m, n, B, nrhs, G2, C));
    if (sh) LQ_TRY(comm_allreduce_sum(c, G2, (long long)n * (n + nrhs)));
    LQ_TRY(launch<chol_upper128_kernel>(c, 1, 1024, 0, c->stream, 0, G2, n, w.R2.as<double>(), stat.as<double>() + 2));
    LQ_TRY(launch_triu_inverse(c, w.R2.as<double>(), n, w.R2inv.as<double>()));
    // the n x nrhs tail
    LQ_TRY(gemm(c, true, false, n, nrhs, n, 1.0, w.R2inv.as<double>(), n, C, nrhs, 0.0, w.Y.as<double>(), nrhs));
    LQ_TRY(gemm(c, false, false, n, nrhs, n, 1.0, w.R2inv.as<double>(), n, w.Y.as<double>(), nrhs, 0.0, w.Z.as<double>(), nrhs));
    LQ_TRY(gemm(c, false, false, n, nrhs, n, 1.0, w.Rinv.as<double>(), n, w.Z.as<double>(), nrhs, 0.0, X, nrhs));
    return read_cholqr_status(c, stat.as<double>(), w, n, st);
}

// Row-sharded fallback (communication-avoiding least squares): the Householder reduction tree of [A_local | B_local], the
// all-gathered local R factors reduced again; the top n rows of the result are [R | Q^T B].  Backward stable for any cond(A).
static int lstsq_tree_sharded(Ctx* c, const double* A, long long m, int n, const double* B, int nrhs, double* X, int* info) {
    const int w = n + nrhs;
    const size_t ww = sizeof(double) * (size_t)w * w;
    DevBuf AB, Rall, Rf;
    LQ_TRY(AB.alloc(c, sizeof(double) * (size_t)m * w));
    LQ_TRY(Rall.alloc(c, ww * c->nranks));
    LQ_TRY(Rf.alloc(c, ww));
    LQ_CUDA(c, cudaMemcpy2DAsync(AB.p, sizeof(double) * w, A, sizeof(double) * n, sizeof(double) * n, (size_t)m,
                                 cudaMemcpyDeviceToDevice, c->stream));
    LQ_CUDA(c, cudaMemcpy2DAsync(AB.as<double>() + n, sizeof(double) * w, B, sizeof(double) * nrhs, sizeof(double) * nrhs,
                                 (size_t)m, cudaMemcpyDeviceToDevice, c->stream));
    LQ_TRY(sharded_rfactor(c, AB.as<double>(), w, m, w, Rall.as<double>(), Rf.as<double>()));
    return launch<backsub_aug_kernel>(c, 1, 128, 0, c->stream, 0, Rf.as<double>(), w, n, nrhs, X, info);
}

int lstsq_tsqr_local(Ctx* c, const double* A, long long m, int n, const double* B, int nrhs, double* X, int* info, bool sharded) {
    const bool sh = sharded && c->nranks > 1;
    // as in tsqr_local, a row-sharded call validates only what every rank sees alike; the rank-local row count goes through the
    // all-reduced "short rank" count
    LQ_REQUIRE(c, n >= 1 && nrhs >= 1 && m >= 1 && (sh || m >= n), LQ_ERR_SHAPE,
               "lstsq_tsqr needs m >= n >= 1 and nrhs >= 1 (got %lld x %d, %d rhs)", m, n, nrhs);
    LQ_REQUIRE(c, m < (1LL << 31), LQ_ERR_SHAPE, "lstsq_tsqr: more than 2^31 rows per device not supported");
    LQ_REQUIRE(c, A && B && X && info, LQ_ERR_ARG, "lstsq_tsqr: null pointer");
    LQ_REQUIRE(c, !sh || n <= 128, LQ_ERR_UNSUPPORTED, "lstsq_tsqr (sharded) supports n <= 128 (got %d)", n);
    const int w = n + nrhs;
    CholQrStatus st;
    bool have_status = false;
    if (n <= 128 && !c->env_tsqr_householder && (sh || m >= 4LL * n)) {
        LQ_TRY(lstsq_cholqr2(c, A, m, n, B, nrhs, X, sh, m < w ? 1.0 : 0.0, &st));
        if (st.ok()) {
            LQ_CUDA(c, cudaMemsetAsync(info, 0, sizeof(int), c->stream));
            return LQ_OK;
        }
        have_status = true;
    }
    // one GPU: the Householder least-squares route of lq_lstsq_householder_batched_info (any n, any conditioning)
    if (!sh) return lstsq_hh_batched_stream(c, c->stream, A, B, 1, (int)m, n, nrhs, X, info);
    LQ_REQUIRE(c, w <= 128, LQ_ERR_UNSUPPORTED,
               "lstsq_tsqr (sharded, n + nrhs = %d > 128): too ill-conditioned for CholeskyQR2, and the reflector tree of [A | B] "
               "supports n + nrhs <= 128", w);
    if (!have_status) LQ_TRY(count_short_ranks(c, m < w ? 1.0 : 0.0, &st.ranks_short));
    LQ_REQUIRE(c, st.ranks_short == 0.0, LQ_ERR_SHAPE,
               "lstsq_tsqr (sharded, reflector path): %d rank(s) hold fewer than n + nrhs = %d rows; re-shard the rows",
               (int)st.ranks_short, w);
    return lstsq_tree_sharded(c, A, m, n, B, nrhs, X, info);
}

}  // namespace lq

using namespace lq;

extern "C" {

int lq_tsqr_dev(lq_ctx* h, const double* A, int64_t m, int n, double* Q, double* R) {
    Ctx* c = as_ctx(h);
    if (!c) return LQ_ERR_ARG;
    LQ_CUDA(c, cudaSetDevice(c->device));
    return tsqr_local(c, A, m, n, Q, R, false);
}
int lq_tsqr_sharded_dev(lq_ctx* h, const double* A, int64_t m, int n, double* Q, double* R) {
    Ctx* c = as_ctx(h);
    if (!c) return LQ_ERR_ARG;
    LQ_CUDA(c, cudaSetDevice(c->device));
    return tsqr_local(c, A, m, n, Q, R, true);
}

int lq_lstsq_tsqr_dev(lq_ctx* h, const double* A, int64_t m, int n, const double* B, int nrhs, double* X, int32_t* info) {
    Ctx* c = as_ctx(h);
    if (!c) return LQ_ERR_ARG;
    LQ_CUDA(c, cudaSetDevice(c->device));
    return lstsq_tsqr_local(c, A, m, n, B, nrhs, X, info, false);
}
int lq_lstsq_tsqr_sharded_dev(lq_ctx* h, const double* A, int64_t m, int n, const double* B, int nrhs, double* X, int32_t* info) {
    Ctx* c = as_ctx(h);
    if (!c) return LQ_ERR_ARG;
    LQ_CUDA(c, cudaSetDevice(c->device));
    return lstsq_tsqr_local(c, A, m, n, B, nrhs, X, info, true);
}

}  // extern "C"

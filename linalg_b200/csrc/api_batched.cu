// Batched QR / least-squares / SVD: the dispatchers and the device-pointer entry points (a1-a5 of SURVEY.md section 8).
// The host-pointer entry points are in api_host.cu.
#include "../../include/linalg_b200.h"
#include "batched_qr32.cuh"
#include "batched_qr32_c8.cuh"
#include "batched_small.cuh"
#include "batched_svd_small.cuh"
#include "ctx.cuh"
#include "ops.cuh"

namespace lq {

// The one-CTA kernels take 32 x 32 matrices too, so the batched 32 x 32 kernels need no case of their own here.
bool hh_qr_batched_one_launch(Ctx* c, int m, int n) {
    return small_hh_smem_doubles(m, n, 0) * sizeof(double) <= (size_t)c->max_smem;
}

int hh_qr_batched_stream(Ctx* c, cudaStream_t st, const double* A, long long batch, int m, int n, double* Q,
                         double* R, bool qr32) {
    if (batch == 0) return LQ_OK;
    if (!hh_qr_batched_one_launch(c, m, n)) {
        // too large for one CTA: blocked path, matrix by matrix (stream `st` must be the context stream)
        for (long long b = 0; b < batch; ++b)
            LQ_TRY(blocked_householder_qr(c, A + b * (long long)m * n, m, n, Q + b * (long long)m * n,
                                          R + b * (long long)n * n));
        return LQ_OK;
    }
    if (m == 32 && n == 32 && qr32) {
        // lane = column, four matrices per warp, left-looking panels, Q formation on DMMA, one 8-warp CTA per SM
        constexpr int WARPS = 8;
        const size_t smem = (size_t)WARPS * Col8::WARP_DOUBLES * sizeof(double);
        return launch<hh_qr32_c8_kernel<WARPS, 1>>(c, (batch + 4 * WARPS - 1) / (4 * WARPS), WARPS * 32, smem, st, (int)smem, A,
                                                   Q, R, batch);
    }
    const size_t smem = small_hh_smem_doubles(m, n, 0) * sizeof(double);
    return launch<small_hh_kernel<0>>(c, batch, 256, smem, st, c->max_smem, A, nullptr, Q, R, nullptr, nullptr, m, n, 0);
}

bool mgs_qr_batched_one_launch(Ctx* c, int m, int n) {
    return small_mgs_smem_doubles(m, n, 0) * sizeof(double) <= (size_t)c->max_smem;
}

int mgs_qr_batched_stream(Ctx* c, cudaStream_t st, const double* A, long long batch, int m, int n, int reorth,
                          double* Q, double* R, int* info) {
    if (batch == 0) return LQ_OK;
    if (!mgs_qr_batched_one_launch(c, m, n)) {
        for (long long b = 0; b < batch; ++b)
            LQ_TRY(large_mgs_qr(c, A + b * (long long)m * n, m, n, reorth, Q + b * (long long)m * n,
                                R + b * (long long)n * n, info ? info + b : nullptr));
        return LQ_OK;
    }
    if (m == 32 && n == 32) {
        using D = Dist32<2, 4>;
        constexpr int WARPS = 2;
        const long long per_block = (long long)WARPS * D::MPW;
        return launch<mgs_qr32_kernel<2, 4, WARPS, 4>>(c, (batch + per_block - 1) / per_block, WARPS * 32,
                                                       (size_t)per_block * D::MGS_DOUBLES * sizeof(double), st, 0, A, Q, R, info,
                                                       batch, reorth);
    }
    const size_t smem = small_mgs_smem_doubles(m, n, 0) * sizeof(double);
    return launch<small_mgs_kernel<0>>(c, batch, 256, smem, st, c->max_smem, A, nullptr, Q, R, nullptr, info, m, n, 0, reorth);
}

bool lstsq_hh_batched_one_launch(Ctx* c, int m, int n, int nrhs) {
    return lstsq_tile_kernel_supported(m, n, nrhs) || lstsq_stream_kernel_supported(m, n, nrhs) ||
           small_hh_smem_doubles(m, n, nrhs) * sizeof(double) <= (size_t)c->max_smem;
}

// info (device, may be null): per system 0, or 1 + the first column whose R[j][j] is exactly 0 (np.linalg.solve raises
// LinAlgError("Singular matrix") there, linalg/qr.py:134); every route writes it
int lstsq_hh_batched_stream(Ctx* c, cudaStream_t st, const double* A, const double* B, long long batch, int m, int n,
                            int nrhs, double* X, int* info) {
    if (batch == 0) return LQ_OK;
    if (!lstsq_hh_batched_one_launch(c, m, n, nrhs)) {
        for (long long b = 0; b < batch; ++b)
            LQ_TRY(large_lstsq_householder(c, A + b * (long long)m * n, B + b * (long long)m * nrhs, m, n, nrhs,
                                           X + b * (long long)n * nrhs, info ? info + b : nullptr));
        return LQ_OK;
    }
    int rc = lstsq_tile_kernel_launch(c, st, A, B, batch, m, n, nrhs, X, info, 2);
    if (rc != LQ_ERR_UNSUPPORTED) return rc;
    rc = lstsq_stream_kernel_launch(c, st, A, B, batch, m, n, nrhs, X, info);
    if (rc != LQ_ERR_UNSUPPORTED) return rc;
    const size_t smem = small_hh_smem_doubles(m, n, nrhs) * sizeof(double);
    return launch<small_hh_kernel<1>>(c, batch, 256, smem, st, c->max_smem, A, B, nullptr, nullptr, X, info, m, n, nrhs);
}

bool lstsq_mgs_batched_one_launch(Ctx* c, int m, int n, int nrhs) {
    return lstsq_tile_kernel_supported(m, n, nrhs) || small_mgs_smem_doubles(m, n, nrhs) * sizeof(double) <= (size_t)c->max_smem;
}

int lstsq_mgs_batched_stream(Ctx* c, cudaStream_t st, const double* A, const double* B, long long batch, int m, int n,
                             int nrhs, double* X, int* info) {
    if (batch == 0) return LQ_OK;
    if (!lstsq_mgs_batched_one_launch(c, m, n, nrhs)) {
        for (long long b = 0; b < batch; ++b)
            LQ_TRY(large_lstsq_mgs(c, A + b * (long long)m * n, B + b * (long long)m * nrhs, m, n, nrhs,
                                   X + b * (long long)n * nrhs, info ? info + b : nullptr));
        return LQ_OK;
    }
    // Only X and the dependence report are observable (linalg/qr.py:103-119): the solution is the one of the
    // Householder entry point and |R[j][j]| does not depend on how the QR factorisation was computed.
    {
        const int rc = lstsq_tile_kernel_launch(c, st, A, B, batch, m, n, nrhs, X, info, 1);
        if (rc != LQ_ERR_UNSUPPORTED) return rc;
    }
    const size_t smem = small_mgs_smem_doubles(m, n, nrhs) * sizeof(double);
    return launch<small_mgs_kernel<1>>(c, batch, 256, smem, st, c->max_smem, A, B, nullptr, nullptr, X, info, m, n, nrhs, 0);
}

// rank (device): #(s > tol) per matrix.  The route depends on (m, n) only, so a matrix's result does not depend on the batch
// it is in: the warp-per-matrix kernel, or the single-matrix pipeline matrix by matrix (bitwise svd(A[b]); stream `st` must
// then be the context stream).
int svd_batched_stream(Ctx* c, cudaStream_t st, const double* A, long long batch, int m, int n, double tol, double* U,
                       double* s, double* Vt, int* rank) {
    if (batch == 0) return LQ_OK;
    if (svd_small_supported(m, n)) {
        constexpr int WARPS = 4;
        const size_t smem = (size_t)WARPS * SvdSmall::WARP_DOUBLES * sizeof(double);
        return launch<svd_small_kernel<WARPS>>(c, (batch + WARPS - 1) / WARPS, WARPS * 32, smem, st, (int)smem, A, batch, m, n,
                                               tol, U, s, Vt, rank);
    }
    for (long long b = 0; b < batch; ++b)
        LQ_TRY(svd_gram_local(c, A + b * (long long)m * n, m, n, tol, U + b * (long long)m * n, s + b * (long long)n,
                              Vt + b * (long long)n * n, nullptr, false, rank + b));
    return LQ_OK;
}

}  // namespace lq

using namespace lq;

extern "C" {

int lq_householder_qr_batched_dev(lq_ctx* h, const double* A, int64_t batch, int m, int n, double* Q, double* R,
                                  int variant) {
    Ctx* c = as_ctx(h);
    LQ_ARGS_QR(c, A, batch, m, n);
    LQ_REQUIRE(c, m >= n, LQ_ERR_SHAPE, "householder_qr needs m >= n (got %d x %d), linalg/qr.py:52", m, n);
    LQ_REQUIRE(c, variant == 0, LQ_ERR_ARG, "householder_qr_batched: kernel variant %d does not exist (0 is the only one)",
               variant);
    LQ_CUDA(c, cudaSetDevice(c->device));
    return hh_qr_batched_stream(c, c->stream, A, batch, m, n, Q, R, true);
}

int lq_mgs_qr_batched_dev(lq_ctx* h, const double* A, int64_t batch, int m, int n, int reorth, double* Q, double* R,
                          int32_t* info) {
    Ctx* c = as_ctx(h);
    LQ_ARGS_QR(c, A, batch, m, n);
    LQ_CUDA(c, cudaSetDevice(c->device));
    return mgs_qr_batched_stream(c, c->stream, A, batch, m, n, reorth, Q, R, info);
}

int lq_lstsq_householder_batched_dev(lq_ctx* h, const double* A, const double* B, int64_t batch, int m, int n,
                                     int nrhs, double* X) {
    Ctx* c = as_ctx(h);
    LQ_ARGS_QR(c, A, batch, m, n);
    LQ_REQUIRE(c, m >= n && nrhs >= 1, LQ_ERR_SHAPE, "least squares needs m >= n and nrhs >= 1 (got %d x %d, %d rhs)", m,
               n, nrhs);
    LQ_CUDA(c, cudaSetDevice(c->device));
    return lstsq_hh_batched_stream(c, c->stream, A, B, batch, m, n, nrhs, X);
}

int lq_lstsq_householder_batched_info_dev(lq_ctx* h, const double* A, const double* B, int64_t batch, int m, int n,
                                          int nrhs, double* X, int32_t* info) {
    Ctx* c = as_ctx(h);
    LQ_ARGS_QR(c, A, batch, m, n);
    LQ_REQUIRE(c, m >= n && nrhs >= 1, LQ_ERR_SHAPE, "least squares needs m >= n and nrhs >= 1 (got %d x %d, %d rhs)", m,
               n, nrhs);
    LQ_CUDA(c, cudaSetDevice(c->device));
    return lstsq_hh_batched_stream(c, c->stream, A, B, batch, m, n, nrhs, X, info);
}

int lq_lstsq_mgs_batched_dev(lq_ctx* h, const double* A, const double* B, int64_t batch, int m, int n, int nrhs,
                             double* X, int32_t* info) {
    Ctx* c = as_ctx(h);
    LQ_ARGS_QR(c, A, batch, m, n);
    LQ_REQUIRE(c, nrhs >= 1, LQ_ERR_SHAPE, "nrhs must be >= 1");
    LQ_CUDA(c, cudaSetDevice(c->device));
    return lstsq_mgs_batched_stream(c, c->stream, A, B, batch, m, n, nrhs, X, info);
}

int lq_svd_gram_batched_dev(lq_ctx* h, const double* A, int64_t batch, int m, int n, double tol, double* U, double* s,
                            double* Vt, int32_t* rank) {
    Ctx* c = as_ctx(h);
    LQ_ARGS_QR(c, A, batch, m, n);
    LQ_REQUIRE(c, m >= n, LQ_ERR_SHAPE, "svd_gram needs m >= n (got %d x %d; transpose on the host side, svd.py:37-39)", m, n);
    LQ_CUDA(c, cudaSetDevice(c->device));
    return svd_batched_stream(c, c->stream, A, batch, m, n, tol, U, s, Vt, rank);
}

}  // extern "C"

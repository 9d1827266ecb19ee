// Batched QR / least-squares / SVD entry points (a1-a5 of SURVEY.md section 8).
#include <algorithm>

#include "../../include/linalg_b200.h"
#include "batched_qr32.cuh"
#include "batched_qr32_c8.cuh"
#include "batched_small.cuh"
#include "batched_svd_small.cuh"
#include "ctx.cuh"
#include "ops.cuh"

namespace lq {

int hh_qr_batched_stream(Ctx* c, cudaStream_t st, const double* A, long long batch, int m, int n, double* Q,
                         double* R, bool qr32) {
    if (batch == 0) return LQ_OK;
    if (m == 32 && n == 32 && qr32) {
        // lane = column, four matrices per warp, left-looking panels, Q formation on DMMA, one 8-warp CTA per SM
        constexpr int WARPS = 8;
        const size_t smem = (size_t)WARPS * Col8::WARP_DOUBLES * sizeof(double);
        return launch<hh_qr32_c8_kernel<WARPS, 1>>(c, (batch + 4 * WARPS - 1) / (4 * WARPS), WARPS * 32, smem, st, (int)smem, A,
                                                   Q, R, batch);
    }
    const size_t smem = small_hh_smem_doubles(m, n, 0) * sizeof(double);
    if (smem <= (size_t)c->max_smem)
        return launch<small_hh_kernel<0>>(c, batch, 256, smem, st, c->max_smem, A, nullptr, Q, R, nullptr, nullptr, m, n, 0);
    // too large for one CTA: blocked path, matrix by matrix (stream `st` must be the context stream)
    for (long long b = 0; b < batch; ++b)
        LQ_TRY(blocked_householder_qr(c, A + b * (long long)m * n, m, n, Q + b * (long long)m * n,
                                      R + b * (long long)n * n));
    return LQ_OK;
}

int mgs_qr_batched_stream(Ctx* c, cudaStream_t st, const double* A, long long batch, int m, int n, int reorth,
                          double* Q, double* R, int* info) {
    if (batch == 0) return LQ_OK;
    if (m == 32 && n == 32) {
        using D = Dist32<2, 4>;
        constexpr int WARPS = 2;
        const long long per_block = (long long)WARPS * D::MPW;
        return launch<mgs_qr32_kernel<2, 4, WARPS, 4>>(c, (batch + per_block - 1) / per_block, WARPS * 32,
                                                       (size_t)per_block * D::MGS_DOUBLES * sizeof(double), st, 0, A, Q, R, info,
                                                       batch, reorth);
    }
    const size_t smem = small_mgs_smem_doubles(m, n, 0) * sizeof(double);
    if (smem <= (size_t)c->max_smem)
        return launch<small_mgs_kernel<0>>(c, batch, 256, smem, st, c->max_smem, A, nullptr, Q, R, nullptr, info, m, n, 0,
                                           reorth);
    for (long long b = 0; b < batch; ++b)
        LQ_TRY(large_mgs_qr(c, A + b * (long long)m * n, m, n, reorth, Q + b * (long long)m * n,
                            R + b * (long long)n * n, info ? info + b : nullptr));
    return LQ_OK;
}

// info (device, may be null): per system 0, or 1 + the first column whose R[j][j] is exactly 0 (np.linalg.solve raises
// LinAlgError("Singular matrix") there, linalg/qr.py:134); every route writes it
int lstsq_hh_batched_stream(Ctx* c, cudaStream_t st, const double* A, const double* B, long long batch, int m, int n,
                            int nrhs, double* X, int* info) {
    if (batch == 0) return LQ_OK;
    int rc = lstsq_tile_kernel_launch(c, st, A, B, batch, m, n, nrhs, X, info, 2);
    if (rc != LQ_ERR_UNSUPPORTED) return rc;
    rc = lstsq_stream_kernel_launch(c, st, A, B, batch, m, n, nrhs, X, info);
    if (rc != LQ_ERR_UNSUPPORTED) return rc;
    const size_t smem = small_hh_smem_doubles(m, n, nrhs) * sizeof(double);
    if (smem <= (size_t)c->max_smem)
        return launch<small_hh_kernel<1>>(c, batch, 256, smem, st, c->max_smem, A, B, nullptr, nullptr, X, info, m, n, nrhs);
    for (long long b = 0; b < batch; ++b)
        LQ_TRY(large_lstsq_householder(c, A + b * (long long)m * n, B + b * (long long)m * nrhs, m, n, nrhs,
                                       X + b * (long long)n * nrhs, info ? info + b : nullptr));
    return LQ_OK;
}

int lstsq_mgs_batched_stream(Ctx* c, cudaStream_t st, const double* A, const double* B, long long batch, int m, int n,
                             int nrhs, double* X, int* info) {
    if (batch == 0) return LQ_OK;
    // Only X and the dependence report are observable (linalg/qr.py:103-119): the solution is the one of the
    // Householder entry point and |R[j][j]| does not depend on how the QR factorisation was computed.
    {
        const int rc = lstsq_tile_kernel_launch(c, st, A, B, batch, m, n, nrhs, X, info, 1);
        if (rc != LQ_ERR_UNSUPPORTED) return rc;
    }
    const size_t smem = small_mgs_smem_doubles(m, n, nrhs) * sizeof(double);
    if (smem <= (size_t)c->max_smem)
        return launch<small_mgs_kernel<1>>(c, batch, 256, smem, st, c->max_smem, A, B, nullptr, nullptr, X, info, m, n, nrhs,
                                           0);
    for (long long b = 0; b < batch; ++b)
        LQ_TRY(large_lstsq_mgs(c, A + b * (long long)m * n, B + b * (long long)m * nrhs, m, n, nrhs,
                               X + b * (long long)n * nrhs, info ? info + b : nullptr));
    return LQ_OK;
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

// ------------------------------------------------------------------ host-pointer pipelines
// Chunks of the batch flow through two lanes (stream + device buffers each): H2D, kernel and D2H
// of neighbouring chunks overlap on the copy engines.  With pinned host buffers the copies are
// truly asynchronous; pageable buffers still work (the runtime stages them).
static long long pick_chunk(long long batch, size_t bytes_per_item) {
    const size_t target = (size_t)192 << 20;  // ~192 MiB of device traffic per chunk
    long long ch = (long long)std::max<size_t>(1, target / std::max<size_t>(1, bytes_per_item));
    return std::min(batch, ch);
}

// out_c / hOc: a third floating-point output (the singular values of the SVD), 0 / nullptr for the others
template <typename Fn>
static int run_chunked(Ctx* c, long long batch, size_t in_a, size_t in_b, size_t out_a, size_t out_b, size_t out_i,
                       const void* hA, const void* hB, void* hOa, void* hOb, void* hInfo, size_t out_c, void* hOc, Fn&& fn) {
    if (batch == 0) return LQ_OK;
    LQ_CUDA(c, cudaSetDevice(c->device));
    const long long chunk = pick_chunk(batch, in_a + in_b + out_a + out_b + out_i + out_c);
    DevBuf dA[2], dB[2], dOa[2], dOb[2], dI[2], dOc[2];
    for (int l = 0; l < 2; ++l) {
        LQ_TRY(dA[l].alloc(c, in_a * chunk, c->lane[l]));
        LQ_TRY(dB[l].alloc(c, in_b * chunk, c->lane[l]));
        LQ_TRY(dOa[l].alloc(c, out_a * chunk, c->lane[l]));
        LQ_TRY(dOb[l].alloc(c, out_b * chunk, c->lane[l]));
        LQ_TRY(dI[l].alloc(c, out_i * chunk, c->lane[l]));
        if (out_c) LQ_TRY(dOc[l].alloc(c, out_c * chunk, c->lane[l]));
    }
    int k = 0;
    for (long long off = 0; off < batch; off += chunk, ++k) {
        const int l = k & 1;
        cudaStream_t st = c->lane[l];
        const long long cnt = std::min(chunk, batch - off);
        LQ_CUDA(c, cudaMemcpyAsync(dA[l].p, (const char*)hA + off * in_a, in_a * cnt, cudaMemcpyHostToDevice, st));
        if (in_b)
            LQ_CUDA(c, cudaMemcpyAsync(dB[l].p, (const char*)hB + off * in_b, in_b * cnt, cudaMemcpyHostToDevice, st));
        LQ_TRY(fn(st, cnt, dA[l].p, dB[l].p, dOa[l].p, dOb[l].p, dI[l].p, dOc[l].p));
        if (out_a)
            LQ_CUDA(c, cudaMemcpyAsync((char*)hOa + off * out_a, dOa[l].p, out_a * cnt, cudaMemcpyDeviceToHost, st));
        if (out_b)
            LQ_CUDA(c, cudaMemcpyAsync((char*)hOb + off * out_b, dOb[l].p, out_b * cnt, cudaMemcpyDeviceToHost, st));
        if (out_i && hInfo)
            LQ_CUDA(c, cudaMemcpyAsync((char*)hInfo + off * out_i, dI[l].p, out_i * cnt, cudaMemcpyDeviceToHost, st));
        if (out_c)
            LQ_CUDA(c, cudaMemcpyAsync((char*)hOc + off * out_c, dOc[l].p, out_c * cnt, cudaMemcpyDeviceToHost, st));
    }
    for (int l = 0; l < 2; ++l) LQ_CUDA(c, cudaStreamSynchronize(c->lane[l]));
    return LQ_OK;
}

static bool fits_small(Ctx* c, size_t doubles) { return doubles * sizeof(double) <= (size_t)c->max_smem; }

}  // namespace lq

using namespace lq;

#define LQ_ARGS_QR(c, A, batch, m, n)                                                                       \
    LQ_REQUIRE(c, c != nullptr, LQ_ERR_ARG, "null context");                                               \
    LQ_REQUIRE(c, batch >= 0 && m >= 1 && n >= 1, LQ_ERR_SHAPE, "bad shape batch=%lld m=%d n=%d",        \
               (long long)batch, m, n);                                                                    \
    LQ_REQUIRE(c, batch == 0 || A != nullptr, LQ_ERR_ARG, "null input pointer")

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

int lq_householder_qr_batched(lq_ctx* h, const double* A, int64_t batch, int m, int n, double* Q, double* R) {
    Ctx* c = as_ctx(h);
    LQ_ARGS_QR(c, A, batch, m, n);
    LQ_REQUIRE(c, m >= n, LQ_ERR_SHAPE, "householder_qr needs m >= n (got %d x %d), linalg/qr.py:52", m, n);
    const size_t mn = (size_t)m * n * 8, nn = (size_t)n * n * 8;
    if (!(m == 32 && n == 32) && !fits_small(c, small_hh_smem_doubles(m, n, 0))) {
        // large matrices: one at a time through the blocked path on the context stream
        for (int64_t b = 0; b < batch; ++b)
            LQ_TRY(lq_householder_qr(h, A + b * (size_t)m * n, m, n, Q + b * (size_t)m * n, R + b * (size_t)n * n));
        return LQ_OK;
    }
    return run_chunked(c, batch, mn, 0, mn, nn, 0, A, nullptr, Q, R, nullptr, 0, nullptr,
                       [&](cudaStream_t st, long long cnt, void* dA, void*, void* dQ, void* dR, void*, void*) {
                           return hh_qr_batched_stream(c, st, (const double*)dA, cnt, m, n, (double*)dQ, (double*)dR, true);
                       });
}

int lq_mgs_qr_batched_dev(lq_ctx* h, const double* A, int64_t batch, int m, int n, int reorth, double* Q, double* R,
                          int32_t* info) {
    Ctx* c = as_ctx(h);
    LQ_ARGS_QR(c, A, batch, m, n);
    LQ_CUDA(c, cudaSetDevice(c->device));
    return mgs_qr_batched_stream(c, c->stream, A, batch, m, n, reorth, Q, R, info);
}

int lq_mgs_qr_batched(lq_ctx* h, const double* A, int64_t batch, int m, int n, int reorth, double* Q, double* R,
                      int32_t* info) {
    Ctx* c = as_ctx(h);
    LQ_ARGS_QR(c, A, batch, m, n);
    const size_t mn = (size_t)m * n * 8, nn = (size_t)n * n * 8;
    if (!(m == 32 && n == 32) && !fits_small(c, small_mgs_smem_doubles(m, n, 0))) {
        for (int64_t b = 0; b < batch; ++b)
            LQ_TRY(lq_mgs_qr(h, A + b * (size_t)m * n, m, n, reorth, Q + b * (size_t)m * n, R + b * (size_t)n * n,
                             info ? info + b : nullptr));
        return LQ_OK;
    }
    return run_chunked(c, batch, mn, 0, mn, nn, sizeof(int32_t), A, nullptr, Q, R, info, 0, nullptr,
                       [&](cudaStream_t st, long long cnt, void* dA, void*, void* dQ, void* dR, void* dI, void*) {
                           return mgs_qr_batched_stream(c, st, (const double*)dA, cnt, m, n, reorth, (double*)dQ,
                                                        (double*)dR, (int*)dI);
                       });
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

static int lstsq_hh_host(lq_ctx* h, const double* A, const double* B, int64_t batch, int m, int n, int nrhs, double* X,
                         int32_t* info);

int lq_lstsq_householder_batched(lq_ctx* h, const double* A, const double* B, int64_t batch, int m, int n, int nrhs,
                                 double* X) {
    return lstsq_hh_host(h, A, B, batch, m, n, nrhs, X, nullptr);
}
int lq_lstsq_householder_batched_info(lq_ctx* h, const double* A, const double* B, int64_t batch, int m, int n, int nrhs,
                                      double* X, int32_t* info) {
    return lstsq_hh_host(h, A, B, batch, m, n, nrhs, X, info);
}

static int lstsq_hh_host(lq_ctx* h, const double* A, const double* B, int64_t batch, int m, int n, int nrhs, double* X,
                         int32_t* info) {
    Ctx* c = as_ctx(h);
    LQ_ARGS_QR(c, A, batch, m, n);
    LQ_REQUIRE(c, m >= n && nrhs >= 1, LQ_ERR_SHAPE, "least squares needs m >= n and nrhs >= 1 (got %d x %d, %d rhs)", m,
               n, nrhs);
    const size_t mn = (size_t)m * n * 8, mk = (size_t)m * nrhs * 8, nk = (size_t)n * nrhs * 8;
    if (!fits_small(c, small_hh_smem_doubles(m, n, nrhs)) && !lstsq_stream_kernel_supported(m, n, nrhs) &&
        !lstsq_tile_kernel_supported(m, n, nrhs)) {
        LQ_CUDA(c, cudaSetDevice(c->device));
        for (int64_t b = 0; b < batch; ++b) {
            DevBuf dA, dB, dX, dI;
            LQ_TRY(dA.alloc(c, mn));
            LQ_TRY(dB.alloc(c, mk));
            LQ_TRY(dX.alloc(c, nk));
            if (info) LQ_TRY(dI.alloc(c, 16));
            LQ_CUDA(c, cudaMemcpyAsync(dA.p, A + b * (size_t)m * n, mn, cudaMemcpyHostToDevice, c->stream));
            LQ_CUDA(c, cudaMemcpyAsync(dB.p, B + b * (size_t)m * nrhs, mk, cudaMemcpyHostToDevice, c->stream));
            LQ_TRY(large_lstsq_householder(c, dA.as<double>(), dB.as<double>(), m, n, nrhs, dX.as<double>(),
                                           info ? dI.as<int>() : nullptr));
            LQ_CUDA(c, cudaMemcpyAsync(X + b * (size_t)n * nrhs, dX.p, nk, cudaMemcpyDeviceToHost, c->stream));
            if (info) LQ_CUDA(c, cudaMemcpyAsync(info + b, dI.p, 4, cudaMemcpyDeviceToHost, c->stream));
            LQ_CUDA(c, cudaStreamSynchronize(c->stream));
        }
        return LQ_OK;
    }
    return run_chunked(c, batch, mn, mk, nk, 0, info ? sizeof(int32_t) : 0, A, B, X, nullptr, info, 0, nullptr,
                       [&](cudaStream_t st, long long cnt, void* dA, void* dB, void* dX, void*, void* dI, void*) {
                           return lstsq_hh_batched_stream(c, st, (const double*)dA, (const double*)dB, cnt, m, n, nrhs,
                                                          (double*)dX, info ? (int*)dI : nullptr);
                       });
}

int lq_lstsq_mgs_batched_dev(lq_ctx* h, const double* A, const double* B, int64_t batch, int m, int n, int nrhs,
                             double* X, int32_t* info) {
    Ctx* c = as_ctx(h);
    LQ_ARGS_QR(c, A, batch, m, n);
    LQ_REQUIRE(c, nrhs >= 1, LQ_ERR_SHAPE, "nrhs must be >= 1");
    LQ_CUDA(c, cudaSetDevice(c->device));
    return lstsq_mgs_batched_stream(c, c->stream, A, B, batch, m, n, nrhs, X, info);
}

int lq_lstsq_mgs_batched(lq_ctx* h, const double* A, const double* B, int64_t batch, int m, int n, int nrhs, double* X,
                         int32_t* info) {
    Ctx* c = as_ctx(h);
    LQ_ARGS_QR(c, A, batch, m, n);
    LQ_REQUIRE(c, nrhs >= 1, LQ_ERR_SHAPE, "nrhs must be >= 1");
    const size_t mn = (size_t)m * n * 8, mk = (size_t)m * nrhs * 8, nk = (size_t)n * nrhs * 8;
    if (!fits_small(c, small_mgs_smem_doubles(m, n, nrhs)) && !lstsq_tile_kernel_supported(m, n, nrhs)) {
        LQ_CUDA(c, cudaSetDevice(c->device));
        for (int64_t b = 0; b < batch; ++b) {
            DevBuf dA, dB, dX, dI;
            LQ_TRY(dA.alloc(c, mn));
            LQ_TRY(dB.alloc(c, mk));
            LQ_TRY(dX.alloc(c, nk));
            LQ_TRY(dI.alloc(c, 16));
            LQ_CUDA(c, cudaMemcpyAsync(dA.p, A + b * (size_t)m * n, mn, cudaMemcpyHostToDevice, c->stream));
            LQ_CUDA(c, cudaMemcpyAsync(dB.p, B + b * (size_t)m * nrhs, mk, cudaMemcpyHostToDevice, c->stream));
            LQ_TRY(large_lstsq_mgs(c, dA.as<double>(), dB.as<double>(), m, n, nrhs, dX.as<double>(), dI.as<int>()));
            LQ_CUDA(c, cudaMemcpyAsync(X + b * (size_t)n * nrhs, dX.p, nk, cudaMemcpyDeviceToHost, c->stream));
            if (info) LQ_CUDA(c, cudaMemcpyAsync(info + b, dI.p, 4, cudaMemcpyDeviceToHost, c->stream));
            LQ_CUDA(c, cudaStreamSynchronize(c->stream));
        }
        return LQ_OK;
    }
    return run_chunked(c, batch, mn, mk, nk, 0, sizeof(int32_t), A, B, X, nullptr, info, 0, nullptr,
                       [&](cudaStream_t st, long long cnt, void* dA, void* dB, void* dX, void*, void* dI, void*) {
                           return lstsq_mgs_batched_stream(c, st, (const double*)dA, (const double*)dB, cnt, m, n, nrhs,
                                                           (double*)dX, (int*)dI);
                       });
}

int lq_svd_gram_batched_dev(lq_ctx* h, const double* A, int64_t batch, int m, int n, double tol, double* U, double* s,
                            double* Vt, int32_t* rank) {
    Ctx* c = as_ctx(h);
    LQ_ARGS_QR(c, A, batch, m, n);
    LQ_REQUIRE(c, m >= n, LQ_ERR_SHAPE, "svd_gram needs m >= n (got %d x %d; transpose on the host side, svd.py:37-39)", m, n);
    LQ_CUDA(c, cudaSetDevice(c->device));
    return svd_batched_stream(c, c->stream, A, batch, m, n, tol, U, s, Vt, rank);
}

int lq_svd_gram_batched(lq_ctx* h, const double* A, int64_t batch, int m, int n, double tol, double* U, double* s, double* Vt,
                        int32_t* rank) {
    Ctx* c = as_ctx(h);
    LQ_ARGS_QR(c, A, batch, m, n);
    LQ_REQUIRE(c, m >= n, LQ_ERR_SHAPE, "svd_gram needs m >= n (got %d x %d; transpose on the host side, svd.py:37-39)", m, n);
    if (!svd_small_supported(m, n)) {
        // the single-matrix pipeline, one matrix at a time on the context stream
        for (int64_t b = 0; b < batch; ++b)
            LQ_TRY(lq_svd_gram(h, A + b * (size_t)m * n, m, n, tol, U + b * (size_t)m * n, s + b * (size_t)n, Vt + b * (size_t)n * n,
                               rank + b));
        return LQ_OK;
    }
    const size_t mn = (size_t)m * n * 8, nn = (size_t)n * n * 8;
    return run_chunked(c, batch, mn, 0, mn, nn, sizeof(int32_t), A, nullptr, U, Vt, rank, (size_t)n * 8, s,
                       [&](cudaStream_t st, long long cnt, void* dA, void*, void* dU, void* dVt, void* dR, void* dS) {
                           return svd_batched_stream(c, st, (const double*)dA, cnt, m, n, tol, (double*)dU, (double*)dS,
                                                     (double*)dVt, (int*)dR);
                       });
}

}  // extern "C"

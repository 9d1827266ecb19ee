// Host-pointer entry points.  Each one checks its arguments and stages its operands through stage_host: copy in, run
// the device path, copy out, synchronise.
#include <algorithm>
#include <utility>

#include "../../include/linalg_b200.h"
#include "batched_svd_small.cuh"
#include "ops.cuh"

namespace lq {
namespace {

// One host array of an entry point: `count` elements per batch item.  IN arrays are copied to the device before fn
// runs, OUT and OPTIONAL_OUT arrays back to the host after it.  A null OPTIONAL_OUT (info, rank) is one the caller does not
// want: nothing is allocated or copied for it and fn receives nullptr.
enum Dir { IN, OUT, OPTIONAL_OUT };

template <typename T, Dir D>
struct HostArray {
    T* host;
    size_t count;
    bool staged() const { return D != OPTIONAL_OUT || host != nullptr; }
};

template <typename T>
HostArray<const T, IN> in(const T* host, size_t count) {
    return {host, count};
}
template <typename T>
HostArray<T, OUT> out(T* host, size_t count) {
    return {host, count};
}
template <typename T>
HostArray<T, OPTIONAL_OUT> optional_out(T* host, size_t count) {
    return {host, count};
}

template <typename... T, typename Fn, size_t... I>
int call_on_device(Fn& fn, cudaStream_t st, long long count, DevBuf* dev, std::index_sequence<I...>) {
    return fn(st, count, static_cast<T*>(dev[I].p)...);
}

// fn(stream, count, device pointers in the order of the arrays) runs the device path on `count` consecutive items.
//   pipelined: chunks of the batch (~192 MiB of device traffic each) alternate between two lanes (a stream and device
//              buffers each), so that H2D, kernel and D2H of neighbouring chunks overlap on the copy engines.  With
//              pinned host buffers the copies are truly asynchronous; pageable buffers still work (the runtime stages
//              them).  fn must run on the stream it is given.
//   serial:    one item at a time on the context stream, all of them in one set of device buffers (stream order makes
//              the reuse safe), for device paths that use the context stream and its side streams.
// Either way the call returns when every output is on the host.
template <typename Fn, typename... T, Dir... D>
int stage_host(Ctx* c, long long batch, bool pipelined, Fn&& fn, HostArray<T, D>... arrays) {
    if (batch == 0) return LQ_OK;
    LQ_CUDA(c, cudaSetDevice(c->device));
    constexpr int K = sizeof...(T);
    char* const host[K] = {(char*)arrays.host...};
    const size_t bytes[K] = {(arrays.staged() ? sizeof(T) * arrays.count : 0)...};
    constexpr bool is_in[K] = {(D == IN)...};
    const int lanes = pipelined ? 2 : 1;
    long long chunk = 1;
    if (pipelined) {
        size_t per_item = 0;
        for (size_t b : bytes) per_item += b;
        chunk = std::min(batch, (long long)std::max<size_t>(1, ((size_t)192 << 20) / std::max<size_t>(1, per_item)));
    }
    auto stream = [&](int l) { return pipelined ? c->lane[l] : c->stream; };
    DevBuf dev[2][K];
    for (int l = 0; l < lanes; ++l)
        for (int i = 0; i < K; ++i)
            if (bytes[i]) LQ_TRY(dev[l][i].alloc(c, bytes[i] * chunk, stream(l)));
    int k = 0;
    for (long long off = 0; off < batch; off += chunk, ++k) {
        const int l = k % lanes;
        const cudaStream_t st = stream(l);
        const long long cnt = std::min(chunk, batch - off);
        for (int i = 0; i < K; ++i)
            if (bytes[i] && is_in[i])
                LQ_CUDA(c, cudaMemcpyAsync(dev[l][i].p, host[i] + off * bytes[i], bytes[i] * cnt, cudaMemcpyHostToDevice, st));
        LQ_TRY(call_on_device<T...>(fn, st, cnt, dev[l], std::index_sequence_for<T...>{}));
        for (int i = 0; i < K; ++i)
            if (bytes[i] && !is_in[i])
                LQ_CUDA(c, cudaMemcpyAsync(host[i] + off * bytes[i], dev[l][i].p, bytes[i] * cnt, cudaMemcpyDeviceToHost, st));
    }
    for (int l = 0; l < lanes; ++l) LQ_CUDA(c, cudaStreamSynchronize(stream(l)));
    return LQ_OK;
}

}  // namespace
}  // namespace lq

using namespace lq;

extern "C" {

int lq_householder_qr_batched(lq_ctx* h, const double* A, int64_t batch, int m, int n, double* Q, double* R) {
    Ctx* c = as_ctx(h);
    LQ_ARGS_QR(c, A, batch, m, n);
    LQ_REQUIRE(c, m >= n, LQ_ERR_SHAPE, "householder_qr needs m >= n (got %d x %d), linalg/qr.py:52", m, n);
    const size_t mn = (size_t)m * n, nn = (size_t)n * n;
    // the per-matrix route calls lq_householder_qr_dev, whose CUDA-graph cache sees the same three buffers every time
    const bool one_launch = hh_qr_batched_one_launch(c, m, n);
    return stage_host(
        c, batch, one_launch,
        [&](cudaStream_t st, long long cnt, const double* dA, double* dQ, double* dR) {
            if (one_launch) return hh_qr_batched_stream(c, st, dA, cnt, m, n, dQ, dR, true);
            return lq_householder_qr_dev(h, dA, m, n, dQ, dR);
        },
        in(A, mn), out(Q, mn), out(R, nn));
}

int lq_householder_qr(lq_ctx* h, const double* A, int m, int n, double* Q, double* R) {
    Ctx* c = as_ctx(h);
    if (!c) return LQ_ERR_ARG;
    LQ_REQUIRE(c, m >= 1 && n >= 1 && m >= n, LQ_ERR_SHAPE, "householder_qr needs m >= n >= 1 (got %d x %d)", m, n);
    LQ_REQUIRE(c, A && Q && R, LQ_ERR_ARG, "null pointer");
    const size_t mn = (size_t)m * n, nn = (size_t)n * n;
    return stage_host(
        c, 1, false,
        [&](cudaStream_t, long long, const double* dA, double* dQ, double* dR) { return lq_householder_qr_dev(h, dA, m, n, dQ, dR); },
        in(A, mn), out(Q, mn), out(R, nn));
}

int lq_mgs_qr_batched(lq_ctx* h, const double* A, int64_t batch, int m, int n, int reorth, double* Q, double* R,
                      int32_t* info) {
    Ctx* c = as_ctx(h);
    LQ_ARGS_QR(c, A, batch, m, n);
    const size_t mn = (size_t)m * n, nn = (size_t)n * n;
    return stage_host(
        c, batch, mgs_qr_batched_one_launch(c, m, n),
        [&](cudaStream_t st, long long cnt, const double* dA, double* dQ, double* dR, int32_t* dI) {
            return mgs_qr_batched_stream(c, st, dA, cnt, m, n, reorth, dQ, dR, dI);
        },
        in(A, mn), out(Q, mn), out(R, nn), optional_out(info, 1));
}

int lq_mgs_qr(lq_ctx* h, const double* A, int m, int n, int reorth, double* Q, double* R, int32_t* info) {
    Ctx* c = as_ctx(h);
    if (!c) return LQ_ERR_ARG;
    LQ_REQUIRE(c, m >= 1 && n >= 1 && A && Q && R, LQ_ERR_SHAPE, "mgs_qr: bad arguments");
    const size_t mn = (size_t)m * n, nn = (size_t)n * n;
    return stage_host(
        c, 1, false,
        [&](cudaStream_t st, long long cnt, const double* dA, double* dQ, double* dR, int32_t* dI) {
            return mgs_qr_batched_stream(c, st, dA, cnt, m, n, reorth, dQ, dR, dI);
        },
        in(A, mn), out(Q, mn), out(R, nn), optional_out(info, 1));
}

int lq_lstsq_householder_batched_info(lq_ctx* h, const double* A, const double* B, int64_t batch, int m, int n, int nrhs,
                                      double* X, int32_t* info) {
    Ctx* c = as_ctx(h);
    LQ_ARGS_QR(c, A, batch, m, n);
    LQ_REQUIRE(c, m >= n && nrhs >= 1, LQ_ERR_SHAPE, "least squares needs m >= n and nrhs >= 1 (got %d x %d, %d rhs)", m,
               n, nrhs);
    const size_t mn = (size_t)m * n, mk = (size_t)m * nrhs, nk = (size_t)n * nrhs;
    return stage_host(
        c, batch, lstsq_hh_batched_one_launch(c, m, n, nrhs),
        [&](cudaStream_t st, long long cnt, const double* dA, const double* dB, double* dX, int32_t* dI) {
            return lstsq_hh_batched_stream(c, st, dA, dB, cnt, m, n, nrhs, dX, dI);
        },
        in(A, mn), in(B, mk), out(X, nk), optional_out(info, 1));
}

int lq_lstsq_householder_batched(lq_ctx* h, const double* A, const double* B, int64_t batch, int m, int n, int nrhs,
                                 double* X) {
    return lq_lstsq_householder_batched_info(h, A, B, batch, m, n, nrhs, X, nullptr);
}

int lq_lstsq_mgs_batched(lq_ctx* h, const double* A, const double* B, int64_t batch, int m, int n, int nrhs, double* X,
                         int32_t* info) {
    Ctx* c = as_ctx(h);
    LQ_ARGS_QR(c, A, batch, m, n);
    LQ_REQUIRE(c, nrhs >= 1, LQ_ERR_SHAPE, "nrhs must be >= 1");
    const size_t mn = (size_t)m * n, mk = (size_t)m * nrhs, nk = (size_t)n * nrhs;
    return stage_host(
        c, batch, lstsq_mgs_batched_one_launch(c, m, n, nrhs),
        [&](cudaStream_t st, long long cnt, const double* dA, const double* dB, double* dX, int32_t* dI) {
            return lstsq_mgs_batched_stream(c, st, dA, dB, cnt, m, n, nrhs, dX, dI);
        },
        in(A, mn), in(B, mk), out(X, nk), optional_out(info, 1));
}

int lq_svd_gram_batched(lq_ctx* h, const double* A, int64_t batch, int m, int n, double tol, double* U, double* s, double* Vt,
                        int32_t* rank) {
    Ctx* c = as_ctx(h);
    LQ_ARGS_QR(c, A, batch, m, n);
    LQ_REQUIRE(c, m >= n, LQ_ERR_SHAPE, "svd_gram needs m >= n (got %d x %d; transpose on the host side, svd.py:37-39)", m, n);
    const size_t mn = (size_t)m * n, nn = (size_t)n * n;
    return stage_host(
        c, batch, svd_small_supported(m, n),
        [&](cudaStream_t st, long long cnt, const double* dA, double* dU, double* ds, double* dVt, int32_t* dr) {
            return svd_batched_stream(c, st, dA, cnt, m, n, tol, dU, ds, dVt, dr);
        },
        in(A, mn), out(U, mn), out(s, (size_t)n), out(Vt, nn), out(rank, 1));
}

int lq_svd_gram(lq_ctx* h, const double* A, int64_t m, int n, double tol, double* U, double* s, double* Vt,
                int* rank_host) {
    Ctx* c = as_ctx(h);
    if (!c) return LQ_ERR_ARG;
    LQ_REQUIRE(c, m >= n && n >= 1, LQ_ERR_SHAPE, "svd_gram needs m >= n >= 1");
    const size_t mn = (size_t)m * n, nn = (size_t)n * n;
    return stage_host(
        c, 1, false,
        [&](cudaStream_t, long long, const double* dA, double* dU, double* ds, double* dVt, int* dr) {
            return svd_gram_local(c, dA, m, n, tol, dU, ds, dVt, nullptr, false, dr);
        },
        in(A, mn), out(U, mn), out(s, (size_t)n), out(Vt, nn), optional_out(rank_host, 1));
}

int lq_tsqr(lq_ctx* h, const double* A, int64_t m, int n, double* Q, double* R) {
    Ctx* c = as_ctx(h);
    if (!c) return LQ_ERR_ARG;
    LQ_REQUIRE(c, m >= n && n >= 1, LQ_ERR_SHAPE, "tsqr needs m >= n >= 1");
    const size_t mn = (size_t)m * n, nn = (size_t)n * n;
    return stage_host(
        c, 1, false,
        [&](cudaStream_t, long long, const double* dA, double* dQ, double* dR) { return tsqr_local(c, dA, m, n, dQ, dR, false); },
        in(A, mn), out(Q, mn), out(R, nn));
}

int lq_lstsq_tsqr(lq_ctx* h, const double* A, int64_t m, int n, const double* B, int nrhs, double* X, int32_t* info) {
    Ctx* c = as_ctx(h);
    if (!c) return LQ_ERR_ARG;
    LQ_REQUIRE(c, m >= n && n >= 1 && nrhs >= 1 && m < (1LL << 31), LQ_ERR_SHAPE,
               "lstsq_tsqr needs 2^31 > m >= n >= 1 and nrhs >= 1 (got %lld x %d, %d rhs)", (long long)m, n, nrhs);
    LQ_REQUIRE(c, A && B && X && info, LQ_ERR_ARG, "lstsq_tsqr: null pointer");
    const size_t mn = (size_t)m * n, mk = (size_t)m * nrhs, nk = (size_t)n * nrhs;
    return stage_host(
        c, 1, false,
        [&](cudaStream_t, long long, const double* dA, const double* dB, double* dX, int32_t* dI) {
            return lstsq_tsqr_local(c, dA, m, n, dB, nrhs, dX, dI, false);
        },
        in(A, mn), in(B, mk), out(X, nk), out(info, 1));
}

}  // extern "C"

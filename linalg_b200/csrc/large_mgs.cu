// Modified Gram-Schmidt (linalg/qr.py:14-49) for a single matrix that does not fit one CTA's
// shared memory.  Right-looking order (identical per-column operation sequence to the reference's
// left-looking loop) on a column-major copy, ONE launch per column: project q_j out of every later
// column; the CTA that owns column j + 1 also normalises it afterwards (it is final then), so the
// next launch finds q_{j+1} ready.  BLAS-2 by nature, L2 resident for typical sizes.
#include "../../include/linalg_b200.h"
#include "ops.cuh"

namespace lq {
namespace {

__device__ __forceinline__ double block_sum256(double v, double* red) {
    v = warp_sum(v);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) red[w] = v;
    __syncthreads();
    double t = (lane < (int)(blockDim.x >> 5)) ? red[lane] : 0.0;
    return warp_sum(t);
}

__global__ void __launch_bounds__(256) transpose_kernel(const double* __restrict__ src, int rows, int cols,
                                                        double* __restrict__ dst /* cols x rows */) {
    __shared__ double tile[32][33];
    const int bx = blockIdx.x * 32, by = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    for (int k = ty; k < 32; k += 8) {
        const int r = by + k, c = bx + tx;
        tile[k][tx] = (r < rows && c < cols) ? src[(size_t)r * cols + c] : 0.0;
    }
    __syncthreads();
    for (int k = ty; k < 32; k += 8) {
        const int c = bx + k, r = by + tx;
        if (c < cols && r < rows) dst[(size_t)c * rows + r] = tile[tx][k];
    }
}

// column j: R[j][j] = ||v||, q = v / ||v||, info
__global__ void __launch_bounds__(256) mgs_norm_kernel(double* __restrict__ At, int m, int n, int j, double* __restrict__ R,
                                                       int* __restrict__ info) {
    __shared__ double red[32];
    double* v = At + (size_t)j * m;
    double p = 0.0;
    for (int i = threadIdx.x; i < m; i += blockDim.x) p = fma(v[i], v[i], p);
    const double nrm = sqrt(block_sum256(p, red));
    if (threadIdx.x == 0) {
        R[(size_t)j * n + j] = nrm;
        if (nrm < kEps && info && *info == 0) *info = j + 1;  // qr.py:40-41
    }
    for (int i = threadIdx.x; i < m; i += blockDim.x) v[i] = v[i] / nrm;  // true division, qr.py:42
}
// columns c > j: r = q_j . a_c ; a_c -= r q_j ; R[j][c] = r      (one CTA per column).  Column j + 1 is final after
// its update: its CTA goes on with R[j+1][j+1] = ||v||, q = v / ||v|| (the work of mgs_norm_kernel for the next step).
__global__ void __launch_bounds__(256) mgs_update_kernel(double* __restrict__ At, int m, int n, int j, double* __restrict__ R,
                                                         int* __restrict__ info) {
    __shared__ double red[32];
    const int c = j + 1 + blockIdx.x;
    const double* q = At + (size_t)j * m;
    double* a = At + (size_t)c * m;
    double p = 0.0;
    for (int i = threadIdx.x; i < m; i += blockDim.x) p = fma(q[i], a[i], p);
    const double r = block_sum256(p, red);
    double p2 = 0.0;
    for (int i = threadIdx.x; i < m; i += blockDim.x) {
        const double v = fma(-r, q[i], a[i]);
        a[i] = v;
        p2 = fma(v, v, p2);
    }
    if (threadIdx.x == 0) R[(size_t)j * n + c] = r;
    if (blockIdx.x == 0) {
        const double nrm = sqrt(block_sum256(p2, red));
        if (threadIdx.x == 0) {
            R[(size_t)c * n + c] = nrm;
            if (nrm < kEps && info && *info == 0) *info = c + 1;  // qr.py:40-41
        }
        for (int i = threadIdx.x; i < m; i += blockDim.x) a[i] = a[i] / nrm;  // true division, qr.py:42 (own writes)
    }
}

}  // namespace

int large_mgs_qr(Ctx* c, const double* A, int m, int n, int reorth, double* Q, double* R, int* info) {
    DevBuf At;
    LQ_TRY(At.alloc(c, sizeof(double) * (size_t)m * n));
    dim3 g1((n + 31) / 32, (m + 31) / 32);
    LQ_TRY(launch<transpose_kernel>(c, g1, 256, 0, c->stream, 0, A, m, n, At.as<double>()));
    LQ_CUDA(c, cudaMemsetAsync(R, 0, sizeof(double) * (size_t)n * n, c->stream));
    if (info) LQ_CUDA(c, cudaMemsetAsync(info, 0, sizeof(int), c->stream));
    for (int sweep = 0; sweep <= (reorth ? 1 : 0); ++sweep) {
        LQ_TRY(launch<mgs_norm_kernel>(c, 1, 256, 0, c->stream, 0, At.as<double>(), m, n, 0, R, info));
        for (int j = 0; j + 1 < n; ++j)
            LQ_TRY(launch<mgs_update_kernel>(c, n - 1 - j, 256, 0, c->stream, 0, At.as<double>(), m, n, j, R, info));
    }
    dim3 g2((m + 31) / 32, (n + 31) / 32);
    return launch<transpose_kernel>(c, g2, 256, 0, c->stream, 0, At.as<double>(), n, m, Q);
}

int large_lstsq_mgs(Ctx* c, const double* A, const double* B, int m, int n, int nrhs, double* X, int* info) {
    DevBuf Qb, Rb;
    LQ_TRY(Qb.alloc(c, sizeof(double) * (size_t)m * n));
    LQ_TRY(Rb.alloc(c, sizeof(double) * (size_t)n * n));
    LQ_TRY(large_mgs_qr(c, A, m, n, 0, Qb.as<double>(), Rb.as<double>(), info));
    LQ_TRY(gemm(c, true, false, n, nrhs, m, 1.0, Qb.as<double>(), n, B, nrhs, 0.0, X, nrhs));  // y = Q^T b  (qr.py:113)
    // one thread per right-hand side at every n (the blocked solve of back_substitute would reorder the sums)
    return backsub_per_column(c, Rb.as<double>(), n, X, nrhs, n, nrhs);
}

}  // namespace lq

using namespace lq;
extern "C" {

int lq_mgs_qr_dev(lq_ctx* h, const double* A, int m, int n, int reorth, double* Q, double* R, int32_t* info) {
    return lq_mgs_qr_batched_dev(h, A, 1, m, n, reorth, Q, R, info);
}

}  // extern "C"

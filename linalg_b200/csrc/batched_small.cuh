// Generic small-matrix kernels: one CTA per matrix, the whole problem resident in shared memory
// (column-major, odd pitch).  These cover every (m, n[, nrhs]) that fits in 227 KB and is not
// served by a specialised kernel; they are the shape-generic implementation of
//   householder_qr              linalg/qr.py:52-100
//   qr (MGS, reorth)            linalg/qr.py:14-49
//   least_squares_householder   linalg/qr.py:122-134   (reflectors applied to [A | B], Q never formed)
//   least_squares_qr            linalg/qr.py:103-119   (y = Q^T b with the ORIGINAL b, then back-substitution)
#pragma once

#include "common.cuh"

namespace lq {

__host__ __device__ inline int small_pitch(int m) { return (m & 1) ? m : m + 1; }  // odd -> conflict-light

// shared-memory doubles needed by the small kernels
__host__ inline size_t small_hh_smem_doubles(int m, int n, int nrhs) {
    return (size_t)small_pitch(m) * (n + nrhs) + 3 * (size_t)n + 64;
}
__host__ inline size_t small_mgs_smem_doubles(int m, int n, int nrhs) {
    return (size_t)small_pitch(m) * (n + nrhs) + (size_t)n * (n + nrhs) + 64;
}

__device__ __forceinline__ double block_sum(double v, double* red /*>=33 doubles*/) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    v = warp_sum(v);
    __syncthreads();  // protect red[] from the previous use
    if (lane == 0) red[warp] = v;
    __syncthreads();
    double t = (lane < nw) ? red[lane] : 0.0;
    t = warp_sum(t);
    return t;  // every thread has the total
}

// mode: 0 = QR (write Q m x n and R n x n), 1 = least squares (write X n x nrhs and, when info is not null, per system
// 0 or 1 + the first column whose R[j][j] is exactly 0: np.linalg.solve raises there, linalg/qr.py:134)
template <int MODE>
__global__ void __launch_bounds__(256)
    small_hh_kernel(const double* __restrict__ A, const double* __restrict__ B, double* __restrict__ Q,
                    double* __restrict__ R, double* __restrict__ X, int* __restrict__ info, int m, int n, int nrhs) {
    extern __shared__ __align__(16) double sm[];
    const int ld = small_pitch(m);
    const int nc = n + nrhs;
    double* W = sm;                      // nc columns, column-major
    double* beta = W + (size_t)ld * nc;  // n
    double* rdiag = beta + n;            // n
    double* vpiv = rdiag + n;            // n   (v0 of every reflector)
    double* red = vpiv + n;              // 64
    const long long b = blockIdx.x;
    const int tid = threadIdx.x, nt = blockDim.x;
    const int lane = tid & 31, warp = tid >> 5, nw = nt >> 5;

    // load (row-major global -> column-major shared)
    {
        const double* Ag = A + b * (long long)m * n;
        for (int e = tid; e < m * n; e += nt) {
            const int i = e / n, c = e - i * n;
            W[(size_t)c * ld + i] = Ag[e];
        }
        if (MODE == 1) {
            const double* Bg = B + b * (long long)m * nrhs;
            for (int e = tid; e < m * nrhs; e += nt) {
                const int i = e / nrhs, c = e - i * nrhs;
                W[(size_t)(n + c) * ld + i] = Bg[e];
            }
        }
    }
    __syncthreads();

    for (int j = 0; j < n; ++j) {
        double* xj = W + (size_t)j * ld;
        double part = 0.0;
        for (int i = j + 1 + tid; i < m; i += nt) part = fma(xj[i], xj[i], part);
        const double sigma = block_sum(part, red);
        const double x0 = xj[j];
        const double nrm = sqrt(fma(x0, x0, sigma));
        const bool skip = nrm < kEps;  // qr.py:79-80
        const double alpha = copysign(nrm, x0);
        const double v0 = x0 + alpha;
        const double bt = skip ? 0.0 : 1.0 / (nrm * fabs(v0));
        __syncthreads();  // everyone has read x0 before it is replaced
        if (tid == 0) {
            beta[j] = bt;
            vpiv[j] = v0;
            rdiag[j] = skip ? x0 : -alpha;
            xj[j] = v0;
        }
        __syncthreads();
        // columns c > j (and the right-hand sides): one warp per column
        for (int c = j + 1 + warp; c < nc; c += nw) {
            double* yc = W + (size_t)c * ld;
            double d = 0.0;
            for (int i = j + lane; i < m; i += 32) d = fma(xj[i], yc[i], d);
            d = warp_sum(d) * bt;
            for (int i = j + lane; i < m; i += 32) yc[i] = fma(-d, xj[i], yc[i]);
        }
        __syncthreads();
    }

    if (MODE == 0) {
        // R (n x n): strict lower triangle exact zeros (qr.py:97)
        double* Rg = R + b * (long long)n * n;
        for (int e = tid; e < n * n; e += nt) {
            const int i = e / n, c = e - i * n;
            Rg[e] = (c > i) ? W[(size_t)c * ld + i] : ((c == i) ? rdiag[i] : 0.0);
        }
        __syncthreads();
        // in-place backward accumulation of the thin Q over the stored reflectors
        for (int j = n - 1; j >= 0; --j) {
            double* vj = W + (size_t)j * ld;
            const double bt = beta[j], v0 = vpiv[j];
            for (int c = j + 1 + warp; c < n; c += nw) {
                double* yc = W + (size_t)c * ld;
                double d = 0.0;
                for (int i = j + 1 + lane; i < m; i += 32) d = fma(vj[i], yc[i], d);
                d = warp_sum(d) * bt;
                for (int i = j + 1 + lane; i < m; i += 32) yc[i] = fma(-d, vj[i], yc[i]);
                if (lane == 0) yc[j] = -d * v0;
            }
            __syncthreads();
            // column j := H_j e_j
            for (int i = tid; i < m; i += nt) {
                double val;
                if (i < j) val = 0.0;
                else if (i == j) val = 1.0 - bt * v0 * v0;
                else val = -bt * v0 * vj[i];
                vj[i] = val;
            }
            __syncthreads();
        }
        double* Qg = Q + b * (long long)m * n;
        for (int e = tid; e < m * n; e += nt) {
            const int i = e / n, c = e - i * n;
            Qg[e] = W[(size_t)c * ld + i];
        }
    } else {
        if (info != nullptr && tid == 0) {
            int bad = 0;
            for (int j = n - 1; j >= 0; --j)
                if (rdiag[j] == 0.0) bad = j + 1;
            info[b] = bad;
        }
        // back-substitution R x = (Q^T B)[:n]; one thread per right-hand side
        for (int k = tid; k < nrhs; k += nt) {
            double* y = W + (size_t)(n + k) * ld;
            for (int i = n - 1; i >= 0; --i) {
                double acc = y[i];
                for (int c = i + 1; c < n; ++c) acc = fma(-W[(size_t)c * ld + i], y[c], acc);
                y[i] = acc / rdiag[i];
            }
        }
        __syncthreads();
        double* Xg = X + b * (long long)n * nrhs;
        for (int e = tid; e < n * nrhs; e += nt) {
            const int i = e / nrhs, k = e - i * nrhs;
            Xg[e] = W[(size_t)(n + k) * ld + i];
        }
    }
}

// Modified Gram-Schmidt, right-looking (identical per-column operation order to qr.py:33-43).
// MODE 0: write Q, R.  MODE 1: least squares, write X (n x nrhs), y = Q^T b on the original b.
template <int MODE>
__global__ void __launch_bounds__(256)
    small_mgs_kernel(const double* __restrict__ A, const double* __restrict__ B, double* __restrict__ Q,
                     double* __restrict__ R, double* __restrict__ X, int* __restrict__ info, int m, int n, int nrhs,
                     int reorth) {
    extern __shared__ __align__(16) double sm[];
    const int ld = small_pitch(m);
    const int nc = n + nrhs;
    double* W = sm;                       // columns of A (then Q) and of B
    double* Rs = W + (size_t)ld * nc;     // n x nc, row-major: R | y
    double* red = Rs + (size_t)n * nc;    // 64
    const long long b = blockIdx.x;
    const int tid = threadIdx.x, nt = blockDim.x;
    const int lane = tid & 31, warp = tid >> 5, nw = nt >> 5;

    {
        const double* Ag = A + b * (long long)m * n;
        for (int e = tid; e < m * n; e += nt) {
            const int i = e / n, c = e - i * n;
            W[(size_t)c * ld + i] = Ag[e];
        }
        if (MODE == 1) {
            const double* Bg = B + b * (long long)m * nrhs;
            for (int e = tid; e < m * nrhs; e += nt) {
                const int i = e / nrhs, c = e - i * nrhs;
                W[(size_t)(n + c) * ld + i] = Bg[e];
            }
        }
        for (int e = tid; e < n * nc; e += nt) Rs[e] = 0.0;
    }
    __syncthreads();

    int bad = 0;
    for (int sweep = 0; sweep <= (reorth ? 1 : 0); ++sweep) {
        for (int j = 0; j < n; ++j) {
            double* qj = W + (size_t)j * ld;
            double part = 0.0;
            for (int i = tid; i < m; i += nt) part = fma(qj[i], qj[i], part);
            const double nrm = sqrt(block_sum(part, red));
            if (nrm < kEps && bad == 0) bad = j + 1;  // qr.py:40-41
            __syncthreads();
            // true division, like the reference's  v / R[j, j]  (qr.py:42): on (near-)triangular inputs the
            // quotient is exactly +-1 and the zeros below stay exact, which tests/test_qr.py:23-47 relies on
            for (int i = tid; i < m; i += nt) qj[i] = qj[i] / nrm;
            if (tid == 0) Rs[(size_t)j * nc + j] = nrm;
            __syncthreads();
            for (int c = j + 1 + warp; c < nc; c += nw) {
                double* yc = W + (size_t)c * ld;
                double d = 0.0;
                for (int i = lane; i < m; i += 32) d = fma(qj[i], yc[i], d);
                d = warp_sum(d);
                if (c < n) {
                    for (int i = lane; i < m; i += 32) yc[i] = fma(-d, qj[i], yc[i]);
                }
                if (lane == 0) Rs[(size_t)j * nc + c] = d;
            }
            __syncthreads();
        }
    }
    if (info != nullptr && tid == 0) info[b] = bad;

    if (MODE == 0) {
        double* Rg = R + b * (long long)n * n;
        for (int e = tid; e < n * n; e += nt) {
            const int i = e / n, c = e - i * n;
            Rg[e] = (c >= i) ? Rs[(size_t)i * nc + c] : 0.0;
        }
        double* Qg = Q + b * (long long)m * n;
        for (int e = tid; e < m * n; e += nt) {
            const int i = e / n, c = e - i * n;
            Qg[e] = W[(size_t)c * ld + i];
        }
    } else {
        for (int k = tid; k < nrhs; k += nt) {
            for (int i = n - 1; i >= 0; --i) {
                double acc = Rs[(size_t)i * nc + n + k];
                for (int c = i + 1; c < n; ++c) acc = fma(-Rs[(size_t)i * nc + c], Rs[(size_t)c * nc + n + k], acc);
                Rs[(size_t)i * nc + n + k] = acc / Rs[(size_t)i * nc + i];
            }
        }
        __syncthreads();
        double* Xg = X + b * (long long)n * nrhs;
        for (int e = tid; e < n * nrhs; e += nt) {
            const int i = e / nrhs, k = e - i * nrhs;
            Xg[e] = Rs[(size_t)i * nc + n + k];
        }
    }
}

}  // namespace lq

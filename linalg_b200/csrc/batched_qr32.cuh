// K2: batched 32x32 MGS QR, matrix distributed over the registers of a lane group.
//
// Reference semantics: linalg/qr.py:14-49 (qr, MGS), applied to every A[b] of a (batch, 32, 32)
// row-major float64 array.
//
// Layout (template P, C): a matrix is spread over L = P * (32 / C) lanes; lane (p, lc) holds
// rows  i = P*ii + p  (ii = 0..32/P-1)  of the C column slots  col(s, lc)  (folded so that
// finished columns retire whole slots: slot s is ascending for even s, descending for odd s).
// With P = 2, C = 4 each lane keeps 4 columns x 16 rows = 64 doubles (128 registers), two
// matrices share a warp, and every column element delivered through shared memory feeds 4 FMAs
// per use; the only cross-lane traffic per column is the column itself, one partner exchange of
// the C partial dot products and one scalar broadcast.  No column norm reduction is needed: the
// owner lane's own dot product IS the sum of squares.
#pragma once

#include "common.cuh"

namespace lq {

template <int P, int C>
struct Dist32 {
    static constexpr int N = 32;
    static constexpr int LC = N / C;    // column lanes
    static constexpr int L = P * LC;    // lanes per matrix
    static constexpr int MPW = 32 / L;  // matrices per warp
    static constexpr int RPL = N / P;   // rows per lane
    static_assert(L <= 32 && L >= 1 && (L & (L - 1)) == 0, "bad distribution");
    // per-matrix shared scratch: two alternating column buffers.  Row lanes (p) and the matrices
    // of a warp are staggered by 4 banks so that the broadcast 16-byte loads of the different
    // (matrix, p) groups of one warp never collide.
    static constexpr int PSTRIDE = RPL + (P > 1 ? 2 : 0);   // doubles between the p sub-rows
    static constexpr int ROWP = P * PSTRIDE;                // doubles per column buffer
    static constexpr int MGS_DOUBLES = 2 * ROWP + (P > 1 ? 4 : 0);
    __device__ __host__ static constexpr int col(int s, int lc) {
        return (s & 1) ? ((s + 1) * LC - 1 - lc) : (s * LC + lc);
    }
    __device__ __host__ static constexpr int owner_slot(int j) { return j / LC; }
    __device__ __host__ static constexpr int owner_lc(int j) {
        return (owner_slot(j) & 1) ? ((owner_slot(j) + 1) * LC - 1 - j) : (j - owner_slot(j) * LC);
    }
};

template <int P, int C>
__device__ __forceinline__ double group_sum(double v) {
    using D = Dist32<P, C>;
#pragma unroll
    for (int o = D::LC; o < D::L; o <<= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// ---------------------------------------------------------------------------------------------
// Modified Gram-Schmidt (right-looking order: per column identical operation sequence to the
// reference's left-looking loop, qr.py:33-43).  Columns are kept unnormalised (v_k) with their
// 1/||v_k||; r_kj = (v_k . a_j)/||v_k||, a_j -= (v_k . a_j)/||v_k||^2 v_k, q_k = v_k/||v_k||.
// info[b] = 1 + first column whose norm fell below 1e-12 (qr.py:40-41), 0 if none.
// reorth: second sweep over Q, R overwritten by the second sweep's R (qr.py:46-47).
// ---------------------------------------------------------------------------------------------
template <int P, int C, int WARPS, int MINB>
__global__ void __launch_bounds__(WARPS * 32, MINB)
    mgs_qr32_kernel(const double* __restrict__ A, double* __restrict__ Q, double* __restrict__ R, int* __restrict__ info,
                    long long batch, int reorth) {
    using D = Dist32<P, C>;
    constexpr int N = 32, RPL = D::RPL, LC = D::LC, L = D::L;
    extern __shared__ __align__(16) double smem[];

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane / L, lm = lane % L, p = lm / LC, lc = lm % LC;
    const long long mat = ((long long)blockIdx.x * WARPS + warp) * D::MPW + g;
    const bool valid = mat < batch;
    const long long matc = valid ? mat : (batch - 1);
    // scratch: two alternating column buffers per matrix; the (matrix, row-lane) groups of a warp are
    // staggered by 4 banks (un-staggered they collide 4-way on every LDS.128)
    double* vb = smem + (size_t)(warp * D::MPW + g) * D::MGS_DOUBLES;

    int colv[C];
#pragma unroll
    for (int s = 0; s < C; ++s) colv[s] = D::col(s, lc);

    double a[C][RPL];
    {
        const double* Ag = A + matc * (N * N) + p * N;
#pragma unroll
        for (int ii = 0; ii < RPL; ++ii)
#pragma unroll
            for (int s = 0; s < C; ++s) a[s][ii] = ld_stream(Ag + ii * (P * N) + colv[s]);
    }
    int bad = 0;
    double* Rg = R + (valid ? mat : 0) * (N * N);

    for (int sweep = 0; sweep <= (reorth ? 1 : 0); ++sweep) {
        double rinvn[C];  // 1/||v_c|| of my finished columns
#pragma unroll
        for (int s = 0; s < C; ++s) rinvn[s] = 1.0;
#pragma unroll
        for (int j = 0; j < N; ++j) {
            const int so = D::owner_slot(j), lo = D::owner_lc(j);
            double* vj = vb + (j & 1) * D::ROWP + p * D::PSTRIDE;
            if (lc == lo) {
#pragma unroll
                for (int ii = 0; ii < RPL; ii += 2)
                    *reinterpret_cast<double2*>(vj + ii) = make_double2(a[so][ii], a[so][ii + 1]);
            }
            __syncwarp();
            double d[C], d2[C], vk[RPL];
#pragma unroll
            for (int s = 0; s < C; ++s) d[s] = 0.0, d2[s] = 0.0;
#pragma unroll
            for (int ii = 0; ii < RPL; ii += 2) {
                const double2 vv = *reinterpret_cast<const double2*>(vj + ii);
                vk[ii] = vv.x;
                vk[ii + 1] = vv.y;
#pragma unroll
                for (int s = so; s < C; ++s) {
                    d[s] = fma(vv.x, a[s][ii], d[s]);
                    d2[s] = fma(vv.y, a[s][ii + 1], d2[s]);
                }
            }
#pragma unroll
            for (int s = so; s < C; ++s) d[s] = group_sum<P, C>(d[s] + d2[s]);
            const double ss = __shfl_sync(0xffffffffu, d[so], lo, L);  // ||v_j||^2
            double rinv;
            // MUFU seed + 2 Newton steps: 2.7e-16 (lq_probe 13..16).  The floor keeps a NaN norm NaN (fmax would turn it
            // into 1e-150 and report the column as dependent, where the reference's R[j, j] < 1e-12 is false and it goes on)
            const double nrm = sqrt_nr_t<2>(ss < 1e-300 ? 1e-300 : ss, rinv);
            if (nrm < kEps && bad == 0) bad = j + 1;
            const double rinv2 = rinv * rinv;
            // R row j: r_jc = d_c / ||v_j|| (c > j), ||v_j|| on the diagonal, 0 left of it
            if (valid && p == 0) {
#pragma unroll
                for (int s = 0; s < C; ++s) {
                    const int c = colv[s];
                    double val = 0.0;
                    if (s >= so) val = (c > j) ? d[s] * rinv : ((c == j) ? nrm : 0.0);
                    st_stream(Rg + j * N + c, val);
                }
            }
#pragma unroll
            for (int s = so; s < C; ++s) {
                const int c = colv[s];
                d[s] = (c > j) ? d[s] * rinv2 : 0.0;
                if (c == j) rinvn[s] = rinv;
            }
#pragma unroll
            for (int ii = 0; ii < RPL; ++ii) {
#pragma unroll
                for (int s = so; s < C; ++s) a[s][ii] = fma(-d[s], vk[ii], a[s][ii]);
            }
        }
        // normalise: q_c = v_c / ||v_c||
#pragma unroll
        for (int s = 0; s < C; ++s)
#pragma unroll
            for (int ii = 0; ii < RPL; ++ii) a[s][ii] *= rinvn[s];
        __syncwarp();
    }

    if (valid) {
        double* Qg = Q + mat * (N * N) + p * N;
#pragma unroll
        for (int ii = 0; ii < RPL; ++ii)
#pragma unroll
            for (int s = 0; s < C; ++s) st_stream(Qg + ii * (P * N) + colv[s], a[s][ii]);
        if (info != nullptr && lm == 0) info[mat] = bad;
    }
}

}  // namespace lq

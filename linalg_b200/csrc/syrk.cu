// G = A^T A for a tall-skinny A (m x n, n <= 128): the Gram matrix of linalg/svd.py:42 and of the two CholeskyQR2 passes
// of the tall-skinny QR (a7), computed as a SYMMETRIC rank-k update -- only the blocks on or above the diagonal are
// multiplied (72 of the 128 m16n8 blocks of a 128 x 128 tile: 56 % of the GEMM's tensor-pipe time), the lower triangle
// is mirrored by the reduction kernel.  SURVEY.md section 8d counts this product as m n^2 flops, not 2 m n^2.
//
// One CTA per SM, each owning a contiguous range of rows (split-K over the whole grid).  A producer warp streams 16-row
// slabs of A with one bulk-async copy per row (TMA engine) into an 8-stage mbarrier ring; because both operands of
// A^T A are the same slab, a stage holds ONE tile (the GEMM kernel holds two).  Eight consumer warps issue
// mma.sync.m16n8k8.f64; the 72 blocks are dealt out so that every warp owns exactly nine: row bands i and 7 - i (16 rows
// each) need 16 - 2 i and 2 + 2 i column blocks, 18 together, shared by a pair of warps.
//
// The strip variant (NS = 32) computes [G | C] = A^T [A | B] for the least-squares pass of the CholeskyQR2 pipeline
// (B m x nrhs, nrhs <= 32): the producer assembles each stage row from two bulk copies (A into columns 0 .. n - 1, B into
// columns 128 .. 128 + nrhs - 1), and every consumer warp also owns the four 16 x 8 blocks of A^T B in the row band it
// already loads (band Q for H = 0, band 7 - Q for H = 1): 13 blocks per warp, 104 in all.  NS = 0 is the plain SYRK.
#include <algorithm>

#include "../../include/linalg_b200.h"
#include "ops.cuh"

namespace lq {

namespace {

constexpr int SBK = 16, SSTAGES = 8;
constexpr int SYRK_THREADS = 288;
constexpr int SYRK_STRIP = 32;  // right-hand-side columns of the strip variant
// stage pitch (doubles): 132 = 4 mod 32 spreads the fragment loads over the banks; the strip variant keeps that residue
template <int NS>
struct SyrkShape {
    static constexpr int SPM = NS == 0 ? 132 : 128 + NS + 4;
    static constexpr int SSTAGE_DOUBLES = SBK * SPM;
    static constexpr int WP = 128 + NS;  // pitch of the per-CTA partial sums
    static constexpr size_t SMEM = (size_t)SSTAGES * SSTAGE_DOUBLES * 8 + 2 * SSTAGES * sizeof(uint64_t) + 16;
};

// the blocks of consumer warp (Q, H): block b lives in row band band(b), column block col(b) (8-column units); blocks
// 9 .. 9 + NS / 8 - 1 are the A^T B blocks of the band the warp's fragment w(b) holds
template <int Q, int H, int NS>
struct SyrkMap {
    static constexpr int NA = H == 0 ? 9 : 7 - 2 * Q;  // blocks of band Q
    static constexpr int NB = 9 + NS / 8;
    __device__ static constexpr int w(int b) { return b < 9 ? (b < NA ? 0 : 1) : H; }
    __device__ static constexpr int band(int b) { return w(b) == 0 ? Q : 7 - Q; }
    __device__ static constexpr int col(int b) {
        return b >= 9 ? 16 + (b - 9) : (H == 0 ? 2 * Q + b : (b < NA ? 2 * Q + 9 + b : 14 - 2 * Q + (b - NA)));
    }
};

template <int Q, int H, int NS>
__device__ __forceinline__ void syrk_consume(const double* tiles, uint64_t* full, uint64_t* empty, int nkt, int lane,
                                             double* __restrict__ Wz) {
    using M = SyrkMap<Q, H, NS>;
    using S = SyrkShape<NS>;
    constexpr int SPM = S::SPM;
    const int gq = lane >> 2, tq = lane & 3;
    double acc[M::NB][4];
#pragma unroll
    for (int b = 0; b < M::NB; ++b)
#pragma unroll
        for (int e = 0; e < 4; ++e) acc[b][e] = 0.0;

    for (int it = 0; it < nkt; ++it) {
        const int s = it % SSTAGES;
        const uint32_t ph = (it / SSTAGES) & 1;
        mbar_wait(&full[s], ph);
        const double* sA = tiles + (size_t)s * S::SSTAGE_DOUBLES;
#pragma unroll
        for (int ks = 0; ks < SBK / 8; ++ks) {
            const int kA = ks * 8 + tq;
            double af[2][4];
#pragma unroll
            for (int w = 0; w < 2; ++w) {
                if (w == 0 && M::NA == 0) continue;
                if (w == 1 && M::NA == 9) continue;
                const int r = 16 * (w == 0 ? Q : 7 - Q) + gq;
                af[w][0] = sA[kA * SPM + r];
                af[w][1] = sA[kA * SPM + r + 8];
                af[w][2] = sA[(kA + 4) * SPM + r];
                af[w][3] = sA[(kA + 4) * SPM + r + 8];
            }
#pragma unroll
            for (int b = 0; b < M::NB; ++b) {
                const int c = 8 * M::col(b) + gq;
                double bf[2];
                bf[0] = sA[kA * SPM + c];
                bf[1] = sA[(kA + 4) * SPM + c];
                dmma_16x8x8(acc[b], af[M::w(b)], bf);
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[s]);
    }
#pragma unroll
    for (int b = 0; b < M::NB; ++b) {
        const int r = 16 * M::band(b) + gq, c = 8 * M::col(b) + 2 * tq;
        *reinterpret_cast<double2*>(Wz + r * S::WP + c) = make_double2(acc[b][0], acc[b][1]);
        *reinterpret_cast<double2*>(Wz + (r + 8) * S::WP + c) = make_double2(acc[b][2], acc[b][3]);
    }
}

// NS = 0: W[z] = partial A^T A (128 x 128).  NS = 32: W[z] = partial A^T [A | B] (128 x 160), B with row stride ldb
template <int NS>
__global__ void __launch_bounds__(SYRK_THREADS, 1)
    syrk_tn_kernel(const double* __restrict__ A, int lda, int n, const double* __restrict__ B, int ldb, int nrhs, int KT,
                   double* __restrict__ W) {
    using S = SyrkShape<NS>;
    constexpr int SSTAGE_DOUBLES = S::SSTAGE_DOUBLES, SPM = S::SPM;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double* tiles = reinterpret_cast<double*>(smem_raw);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + (size_t)SSTAGES * SSTAGE_DOUBLES * 8);
    uint64_t* empty = full + SSTAGES;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    // my k-tiles: the first `rem` CTAs take one more
    const int per = KT / gridDim.x, rem = KT % gridDim.x;
    const int kt0 = blockIdx.x * per + min((int)blockIdx.x, rem);
    const int nkt = per + ((int)blockIdx.x < rem ? 1 : 0);

    if (threadIdx.x == 0) {
        for (int s = 0; s < SSTAGES; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], 8);
        }
        mbar_fence_init();
    }
    if (n < 128 || nrhs < NS) {  // columns n .. 127 (and 128 + nrhs .. 128 + NS - 1) are never written by the row copies
        for (int e = threadIdx.x; e < SSTAGES * SSTAGE_DOUBLES; e += SYRK_THREADS) tiles[e] = 0.0;
        fence_proxy_async();
    }
    __syncthreads();

    if (warp == 8) {
        const uint32_t row_bytes = (uint32_t)n * 8u;
        const uint32_t rhs_bytes = (uint32_t)nrhs * 8u;  // 0 for NS = 0
        for (int it = 0; it < nkt; ++it) {
            const int s = it % SSTAGES;
            const uint32_t ph = (it / SSTAGES) & 1;
            mbar_wait(&empty[s], ph ^ 1);
            double* sA = tiles + (size_t)s * SSTAGE_DOUBLES;
            const long long k0 = (long long)(kt0 + it) * SBK;
            if (lane == 0) mbar_expect_tx(&full[s], SBK * (row_bytes + rhs_bytes));
            __syncwarp();
            if (lane < SBK) bulk_g2s(sA + lane * SPM, A + (k0 + lane) * (long long)lda, row_bytes, &full[s]);
            if (NS > 0 && lane >= SBK)
                bulk_g2s(sA + (lane - SBK) * SPM + 128, B + (k0 + lane - SBK) * (long long)ldb, rhs_bytes, &full[s]);
        }
        return;
    }
    double* Wz = W + (size_t)blockIdx.x * 128 * S::WP;
    switch (warp) {
        case 0: syrk_consume<0, 0, NS>(tiles, full, empty, nkt, lane, Wz); break;
        case 1: syrk_consume<0, 1, NS>(tiles, full, empty, nkt, lane, Wz); break;
        case 2: syrk_consume<1, 0, NS>(tiles, full, empty, nkt, lane, Wz); break;
        case 3: syrk_consume<1, 1, NS>(tiles, full, empty, nkt, lane, Wz); break;
        case 4: syrk_consume<2, 0, NS>(tiles, full, empty, nkt, lane, Wz); break;
        case 5: syrk_consume<2, 1, NS>(tiles, full, empty, nkt, lane, Wz); break;
        case 6: syrk_consume<3, 0, NS>(tiles, full, empty, nkt, lane, Wz); break;
        default: syrk_consume<3, 1, NS>(tiles, full, empty, nkt, lane, Wz); break;
    }
}

// G[r][c] = G[c][r] = sum_z W[z][r][c] (c >= r) + the rows beyond the last whole 16-row slab
__global__ void __launch_bounds__(256)
    syrk_reduce_kernel(const double* __restrict__ W, int splits, const double* __restrict__ Atail, int lda, int tail_rows, int n,
                       double* __restrict__ G, int ldg) {
    const int r = blockIdx.x;
    for (int c = r + threadIdx.x; c < n; c += blockDim.x) {
        double s0 = 0.0, s1 = 0.0;
        int z = 0;
        for (; z + 1 < splits; z += 2) {
            s0 += W[(size_t)z * 16384 + r * 128 + c];
            s1 += W[(size_t)(z + 1) * 16384 + r * 128 + c];
        }
        if (z < splits) s0 += W[(size_t)z * 16384 + r * 128 + c];
        double s = s0 + s1;
        for (int k = 0; k < tail_rows; ++k) s = fma(Atail[(size_t)k * lda + r], Atail[(size_t)k * lda + c], s);
        G[(size_t)r * ldg + c] = s;
        G[(size_t)c * ldg + r] = s;
    }
}

// the strip variant's reduction: G (n x n, both triangles) as above, C[r][k] = sum_z W[z][r][128 + k] + the tail rows
__global__ void __launch_bounds__(256)
    syrk_strip_reduce_kernel(const double* __restrict__ W, int splits, const double* __restrict__ Atail, int lda,
                             const double* __restrict__ Btail, int ldb, int tail_rows, int n, int nrhs, double* __restrict__ G,
                             double* __restrict__ C) {
    constexpr int WP = SyrkShape<SYRK_STRIP>::WP;
    constexpr size_t WZ = (size_t)128 * WP;
    const int r = blockIdx.x;
    for (int c = r + threadIdx.x; c < n; c += blockDim.x) {
        double s0 = 0.0, s1 = 0.0;
        int z = 0;
        for (; z + 1 < splits; z += 2) {
            s0 += W[(size_t)z * WZ + r * WP + c];
            s1 += W[(size_t)(z + 1) * WZ + r * WP + c];
        }
        if (z < splits) s0 += W[(size_t)z * WZ + r * WP + c];
        double s = s0 + s1;
        for (int k = 0; k < tail_rows; ++k) s = fma(Atail[(size_t)k * lda + r], Atail[(size_t)k * lda + c], s);
        G[(size_t)r * n + c] = s;
        G[(size_t)c * n + r] = s;
    }
    for (int c = threadIdx.x; c < nrhs; c += blockDim.x) {
        double s0 = 0.0, s1 = 0.0;
        int z = 0;
        for (; z + 1 < splits; z += 2) {
            s0 += W[(size_t)z * WZ + r * WP + 128 + c];
            s1 += W[(size_t)(z + 1) * WZ + r * WP + 128 + c];
        }
        if (z < splits) s0 += W[(size_t)z * WZ + r * WP + 128 + c];
        double s = s0 + s1;
        for (int k = 0; k < tail_rows; ++k) s = fma(Atail[(size_t)k * lda + r], Btail[(size_t)k * ldb + c], s);
        C[(size_t)r * nrhs + c] = s;
    }
}

int syrk_splits(Ctx* c, int KT) { return (int)std::min<long long>(c->sm_count, std::max(1, KT / 4)); }

}  // namespace

bool syrk_tn_supported(const double* A, int lda, long long m, int n) {
    return n >= 2 && n <= 128 && (n % 2 == 0) && (lda % 2 == 0) && ((reinterpret_cast<uintptr_t>(A) & 15) == 0) &&
           m >= 16LL * 64 && m / SBK < (1LL << 31);
}

// G (n x n, ldg, both triangles) = A^T A, A m x n with row stride lda
int syrk_tn(Ctx* c, const double* A, int lda, long long m, int n, double* G, int ldg) {
    if (!syrk_tn_supported(A, lda, m, n)) return LQ_ERR_UNSUPPORTED;
    const int KT = (int)(m / SBK);
    const int splits = syrk_splits(c, KT);
    constexpr size_t SMEM = SyrkShape<0>::SMEM;
    DevBuf W;
    LQ_TRY(W.alloc(c, sizeof(double) * (size_t)splits * 128 * 128));
    LQ_TRY(launch<syrk_tn_kernel<0>>(c, splits, SYRK_THREADS, SMEM, c->stream, (int)SMEM, A, lda, n, (const double*)nullptr, 0, 0,
                                     KT, W.as<double>()));
    const int tail = (int)(m - (long long)KT * SBK);
    return launch<syrk_reduce_kernel>(c, n, 128, 0, c->stream, 0, W.as<double>(), splits, A + (size_t)KT * SBK * lda, lda, tail, n,
                                      G, ldg);
}

bool syrk_strip_supported(const double* Q, long long m, int n, const double* B, int nrhs) {
    return syrk_tn_supported(Q, n, m, n) && nrhs >= 2 && nrhs <= SYRK_STRIP && nrhs % 2 == 0 &&
           (reinterpret_cast<uintptr_t>(B) & 15) == 0;
}

// G (n x n, both triangles) = Q^T Q and C (n x nrhs) = Q^T B in one pass over Q (m x n) and B (m x nrhs), both densely packed
int syrk_strip_tn(Ctx* c, const double* Q, long long m, int n, const double* B, int nrhs, double* G, double* C) {
    if (!syrk_strip_supported(Q, m, n, B, nrhs)) return LQ_ERR_UNSUPPORTED;
    using S = SyrkShape<SYRK_STRIP>;
    const int KT = (int)(m / SBK);
    const int splits = syrk_splits(c, KT);
    DevBuf W;
    LQ_TRY(W.alloc(c, sizeof(double) * (size_t)splits * 128 * S::WP));
    LQ_TRY(launch<syrk_tn_kernel<SYRK_STRIP>>(c, splits, SYRK_THREADS, S::SMEM, c->stream, (int)S::SMEM, Q, n, n, B, nrhs, nrhs, KT,
                                              W.as<double>()));
    const long long t0 = (long long)KT * SBK;
    return launch<syrk_strip_reduce_kernel>(c, n, 128, 0, c->stream, 0, W.as<double>(), splits, Q + t0 * n, n, B + t0 * nrhs, nrhs,
                                            (int)(m - t0), n, nrhs, G, C);
}

}  // namespace lq

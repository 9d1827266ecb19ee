// Row-major FP64 GEMM  C = alpha * op(A) * op(B) + beta * C  for the blocked-QR / Gram / U=AV paths.
//
// Fast path: 128x128x16 CTA tiles, 8 consumer warps (2 x 4, warp tile 64x32) issuing FP64
// tensor-core MMAs (mma.sync m16n8k8.f64 -> DMMA; tcgen05 has no f64 kind on sm_100a), fed by a
// producer warp that streams operand rows with 1-D bulk-async copies (TMA engine, UBLKCP) into a
// 4-stage mbarrier ring.  Shared tiles are padded (pitch 20 / 132 doubles) so every fragment load
// is bank-conflict free.  Skinny outputs use split-K with a deterministic second-pass reduction.
// Generic path: plain 32x32 tiled kernel for shapes/alignments the fast path does not take.
#include <cuda.h>  // CUtensorMap types only; the encoder is resolved through cudaGetDriverEntryPoint (no -lcuda)

#include <algorithm>

#include "../../include/linalg_b200.h"
#include "ops.cuh"

namespace lq {

namespace {

constexpr int BM = 128, BN = 128, BK = 16, STAGES = 4;
constexpr int PM = 132;   // pitch of an M/N-major tile [k][row] (128 + 4 pad), filled by 16 one-row bulk copies
// A K-major tile [row][k] is 128 rows x 16 doubles = 128 rows x 128 B: ONE 2-D TMA box with the 128-byte
// swizzle (16-byte chunk c of row r lands at chunk c ^ (r & 7)), which makes the DMMA fragment loads
// bank-conflict free without padding.  (128 separate 128-byte bulk copies per stage halved the NN rate.)
constexpr int TILE_BYTES = 17408;   // 17 KiB >= max(128*128, 16*132*8), multiple of 1024 (swizzle alignment)
constexpr int TILE_DOUBLES = TILE_BYTES / 8;
constexpr int GEMM_THREADS = 288;   // 8 consumer warps + 1 producer warp
constexpr size_t GEMM_SMEM = (size_t)STAGES * 2 * TILE_BYTES + 2 * STAGES * sizeof(uint64_t) + 1024;

using EncodeTiledFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                   const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                   CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn tensor_map_encoder() {
    static EncodeTiledFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            p = nullptr;
        return reinterpret_cast<EncodeTiledFn>(p);
    }();
    return fn;
}
// tensor map of a row-major (rows x cols, ld) float64 matrix, box = 128 rows x 16 columns, 128-byte swizzle
int make_kmajor_map(Ctx* c, CUtensorMap* map, const double* base, long long rows, long long cols, long long ld) {
    EncodeTiledFn enc = tensor_map_encoder();
    LQ_REQUIRE(c, enc != nullptr, LQ_ERR_UNSUPPORTED, "cuTensorMapEncodeTiled is not available in this driver");
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * sizeof(double)};
    cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)BM};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 2, const_cast<double*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    LQ_REQUIRE(c, r == CUDA_SUCCESS, LQ_ERR_CUDA_BASE + 1, "cuTensorMapEncodeTiled failed (CUresult %d)", (int)r);
    return LQ_OK;
}

__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
            smem_u32(smem_dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(smem_u32(bar))
        : "memory");
}
// C[i] += v without reading it back: one RED per element, no load round trip in the epilogue.  Every element of C
// is touched by exactly one thread of one CTA, so the result is as deterministic as load-add-store.
__device__ __forceinline__ void red_add(double* p, double v) {
    asm volatile("red.global.add.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory");
}
// the same for a whole row segment: the TMA engine reads the values from shared memory and adds them into global
// memory (SASS UBLKRED.G.S.ADD.F64); bytes % 16 == 0, both addresses 16-byte aligned
__device__ __forceinline__ void bulk_red_add_f64(double* gmem_dst, const double* smem_src, uint32_t bytes) {
    asm volatile("cp.reduce.async.bulk.global.shared::cta.bulk_group.add.f64 [%0], [%1], %2;" ::"l"(gmem_dst),
                 "r"(smem_u32(smem_src)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void consumer_bar_sync() { asm volatile("bar.sync 1, 256;" ::: "memory"); }
constexpr int EPI_PITCH = 136;  // doubles per staged C row: 128 + 8 (a quarter-warp's 16-byte stores hit distinct banks)
static_assert((size_t)BM * EPI_PITCH * 8 <= (size_t)STAGES * 2 * TILE_BYTES, "the staged C tile reuses the operand ring");
// element (r, k) of a swizzled K-major tile (r & 7 must be passed as r7)
__device__ __forceinline__ int sw_idx(int r, int r7, int k) { return r * BK + ((((k >> 1) ^ r7) << 1) | (k & 1)); }

struct GemmArgs {
    const double* A;
    const double* B;
    double* C;       // output (or split-K workspace)
    long long M;
    int N, K;        // K already trimmed to a multiple of BK
    int lda, ldb, ldc;
    double alpha, beta;
    int splits;      // gridDim.z
    long long split_stride;  // elements between split-K slices of the workspace
};

// AT: A is stored K x M (op(A) = A^T)  -> shared tile [k][m]   ("M-major")
// BT: B is stored N x K (op(B) = B^T)  -> shared tile [n][k]   ("K-major")
// 9 warps: registers are granted per 4-warp group, so a 288-thread block is capped at 168 registers/thread; the
// main loop therefore keeps only ONE A fragment live at a time (128 accumulator + 8 + 16 fragment registers).
template <bool AT, bool BT, bool SK = false>  // SK: skinny outputs, bands without valid rows / columns issue no DMMA
__global__ void __launch_bounds__(GEMM_THREADS, 1)
    gemm_dmma_kernel(const GemmArgs g, const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB) {
    extern __shared__ unsigned char smem_dyn[];
    // 1024-byte alignment for the swizzled TMA boxes; the offset is added to the __shared__ symbol itself so that
    // the compiler keeps the shared address space (LDS instead of generic LD)
    unsigned char* smem_raw = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
    double* tiles = reinterpret_cast<double*>(smem_raw);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + (size_t)STAGES * 2 * TILE_BYTES);
    uint64_t* empty = full + STAGES;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long m0 = (long long)blockIdx.y * BM;
    const int n0 = blockIdx.x * BN;
    const int mvalid = (int)min((long long)BM, g.M - m0);
    const int nvalid = min(BN, g.N - n0);

    // split-K range (in k-tiles)
    const int KT = g.K / BK;
    const int per = (KT + g.splits - 1) / g.splits;
    const int kt0 = blockIdx.z * per;
    const int kt1 = min(KT, kt0 + per);
    const int nkt = max(0, kt1 - kt0);

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], 8);
        }
        mbar_fence_init();
    }
    __syncthreads();

    if (warp == 8) {
        // ===================== producer =====================
        // a TMA box always delivers its full size (out-of-range rows arrive as zeros)
        const uint32_t bytesA = AT ? (uint32_t)(BK * mvalid * 8) : (uint32_t)(BM * BK * 8);
        const uint32_t bytesB = BT ? (uint32_t)(BN * BK * 8) : (uint32_t)(BK * nvalid * 8);
        for (int it = 0; it < nkt; ++it) {
            const int s = it % STAGES;
            const uint32_t ph = (it / STAGES) & 1;
            mbar_wait(&empty[s], ph ^ 1);
            double* sA = tiles + (size_t)s * 2 * TILE_DOUBLES;
            double* sB = sA + TILE_DOUBLES;
            const long long k0 = (long long)(kt0 + it) * BK;
            if (lane == 0) mbar_expect_tx(&full[s], bytesA + bytesB);
            __syncwarp();
            if (AT) {
                if (lane < BK) bulk_g2s(sA + lane * PM, g.A + (k0 + lane) * g.lda + m0, mvalid * 8, &full[s]);
            } else {
                if (lane == 0) tma_load_2d(sA, &mapA, (int)k0, (int)m0, &full[s]);
            }
            if (BT) {
                if (lane == 1) tma_load_2d(sB, &mapB, (int)k0, n0, &full[s]);
            } else {
                if (lane >= 16) {
                    const int kk = lane - 16;
                    bulk_g2s(sB + kk * PM, g.B + (k0 + kk) * g.ldb + n0, nvalid * 8, &full[s]);
                }
            }
        }
        return;
    }

    // ===================== consumers =====================
    const int wm = warp >> 2, wn = warp & 3;
    const int gq = lane >> 2, tq = lane & 3;
    double acc[4][4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int e = 0; e < 4; ++e) acc[i][j][e] = 0.0;

    // read-modify-write epilogue ahead: pull my part of the C tile into L2 while the main loop runs
    if (g.splits == 1 && g.beta != 0.0 && g.beta != 1.0) {
#pragma unroll
        for (int im = 0; im < 4; ++im)
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const int r = wm * 64 + im * 16 + gq + half * 8;
                if (r < mvalid && tq == 0) {
                    const double* crow = g.C + (m0 + r) * (long long)g.ldc + n0 + wn * 32;
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(crow));
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(crow + 16));
                }
            }
    }

    // SK instantiation (the V^T C products of the panel chain have 32 valid rows): 16-row / 8-column bands without a
    // valid element issue no DMMA (warp-uniform tests), so a 32 x 96 product costs a fraction of a full tile's pipe time;
    // kept out of the general instantiations, where the predicates cost 9 % on 4096^3
    const int im_lim = min(4, max(0, (mvalid - wm * 64 + 15) >> 4));
    const int jn_lim = min(4, max(0, (nvalid - wn * 32 + 7) >> 3));
    for (int it = 0; it < nkt; ++it) {
        const int s = it % STAGES;
        const uint32_t ph = (it / STAGES) & 1;
        mbar_wait(&full[s], ph);
        const double* sA = tiles + (size_t)s * 2 * TILE_DOUBLES;
        const double* sB = sA + TILE_DOUBLES;
#pragma unroll
        for (int ks = 0; ks < BK / 8; ++ks) {
            double bf[4][2];
            const int kA = ks * 8 + tq;
#pragma unroll
            for (int jn = 0; jn < 4; ++jn) {
                const int c = wn * 32 + jn * 8 + gq;
                if (BT) {
                    bf[jn][0] = sB[sw_idx(c, gq, kA)];
                    bf[jn][1] = sB[sw_idx(c, gq, kA + 4)];
                } else {
                    bf[jn][0] = sB[kA * PM + c];
                    bf[jn][1] = sB[(kA + 4) * PM + c];
                }
            }
#pragma unroll
            for (int im = 0; im < 4; ++im) {
                if (SK && im >= im_lim) continue;
                double af[4];
                const int r = wm * 64 + im * 16 + gq;
                if (AT) {
                    af[0] = sA[kA * PM + r];
                    af[1] = sA[kA * PM + r + 8];
                    af[2] = sA[(kA + 4) * PM + r];
                    af[3] = sA[(kA + 4) * PM + r + 8];
                } else {
                    af[0] = sA[sw_idx(r, gq, kA)];
                    af[1] = sA[sw_idx(r + 8, gq, kA)];
                    af[2] = sA[sw_idx(r, gq, kA + 4)];
                    af[3] = sA[sw_idx(r + 8, gq, kA + 4)];
                }
#pragma unroll
                for (int jn = 0; jn < 4; ++jn)
                    if (!SK || jn < jn_lim) dmma_16x8x8(acc[im][jn], af, bf[jn]);
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[s]);
    }

    // ===================== epilogue =====================
    // Two-phase per 16-row band: all the C loads of the band are issued before any dependent FMA / store,
    // so a thread pays one global round trip per band instead of one per element (the rank-128 update
    // C -= V W spends as long in this epilogue as in its 8 k-tiles otherwise).
    double* Cb = g.C + (long long)blockIdx.z * g.split_stride;
    const bool direct = (g.splits == 1);
    const double alpha = direct ? g.alpha : 1.0;
    const double beta = direct ? g.beta : 0.0;
    const bool vec2 = ((g.ldc & 1) == 0) && ((reinterpret_cast<uintptr_t>(Cb) & 15) == 0);
    if (beta == 1.0 && vec2 && (nvalid & 1) == 0) {
        // In-place accumulation through the TMA engine: the tile is staged in the (now idle) operand ring and leaves
        // as one bulk reduce-add per row, so the 64 scalar REDs per thread disappear from the SM's issue slots and
        // the CTA retires as soon as the engine has read the staging buffer.  One writer per element -> deterministic.
        consumer_bar_sync();  // every consumer warp is done reading the operand stages
        double* stg = tiles;
#pragma unroll
        for (int im = 0; im < 4; ++im)
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const int r = wm * 64 + im * 16 + gq + half * 8;
#pragma unroll
                for (int jn = 0; jn < 4; ++jn) {
                    const int c = wn * 32 + jn * 8 + 2 * tq;
                    *reinterpret_cast<double2*>(stg + r * EPI_PITCH + c) =
                        make_double2(alpha * acc[im][jn][half * 2 + 0], alpha * acc[im][jn][half * 2 + 1]);
                }
            }
        fence_proxy_async();
        consumer_bar_sync();
        if (lane < 16) {
            const int r = warp * 16 + lane;
            if (r < mvalid) bulk_red_add_f64(Cb + (m0 + r) * (long long)g.ldc + n0, stg + r * EPI_PITCH, (uint32_t)nvalid * 8u);
        }
        bulk_commit();
        bulk_wait_read<0>();
        return;
    }
#pragma unroll
    for (int im = 0; im < 4; ++im) {
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const int r = wm * 64 + im * 16 + gq + half * 8;
            if (r >= mvalid) continue;
            double* crow = Cb + (m0 + r) * (long long)g.ldc + n0;
            if (beta == 1.0) {  // accumulate in place: fire-and-forget reductions
#pragma unroll
                for (int jn = 0; jn < 4; ++jn) {
                    const int c = wn * 32 + jn * 8 + 2 * tq;
                    if (c < nvalid) red_add(crow + c, alpha * acc[im][jn][half * 2 + 0]);
                    if (c + 1 < nvalid) red_add(crow + c + 1, alpha * acc[im][jn][half * 2 + 1]);
                }
                continue;
            }
            double cold[4][2];
            if (beta != 0.0) {
#pragma unroll
                for (int jn = 0; jn < 4; ++jn) {
                    const int c = wn * 32 + jn * 8 + 2 * tq;
                    cold[jn][0] = 0.0;
                    cold[jn][1] = 0.0;
                    if (vec2 && c + 1 < nvalid) {
                        const double2 t2 = *reinterpret_cast<const double2*>(crow + c);
                        cold[jn][0] = t2.x;
                        cold[jn][1] = t2.y;
                    } else {
                        if (c < nvalid) cold[jn][0] = crow[c];
                        if (c + 1 < nvalid) cold[jn][1] = crow[c + 1];
                    }
                }
            }
#pragma unroll
            for (int jn = 0; jn < 4; ++jn) {
                const int c = wn * 32 + jn * 8 + 2 * tq;
                double v0 = alpha * acc[im][jn][half * 2 + 0];
                double v1 = alpha * acc[im][jn][half * 2 + 1];
                if (beta != 0.0) {
                    v0 = fma(beta, cold[jn][0], v0);
                    v1 = fma(beta, cold[jn][1], v1);
                }
                if (vec2 && c + 1 < nvalid) {
                    *reinterpret_cast<double2*>(crow + c) = make_double2(v0, v1);
                } else {
                    if (c < nvalid) crow[c] = v0;
                    if (c + 1 < nvalid) crow[c + 1] = v1;
                }
            }
        }
    }
}

// C = alpha * sum_z W[z] + beta * C
__global__ void __launch_bounds__(256) splitk_reduce_kernel(const double* __restrict__ W, int splits, long long stride,
                                                            long long M, int N, double alpha, double beta, double* C,
                                                            int ldc) {
    const long long total = M * N;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const long long i = e / N;
        const int j = (int)(e - i * N);
        double s = 0.0;
        for (int z = 0; z < splits; ++z) s += W[z * stride + e];
        double* cp = C + i * ldc + j;
        double v = alpha * s;
        if (beta != 0.0) v = fma(beta, *cp, v);
        *cp = v;
    }
}

// Generic tiled kernel: any transposition, shape, leading dimension, alignment.
template <bool AT, bool BT>
__global__ void __launch_bounds__(256) gemm_generic_kernel(const double* __restrict__ A, const double* __restrict__ B,
                                                           double* __restrict__ C, long long M, int N, int K, int lda,
                                                           int ldb, int ldc, double alpha, double beta) {
    __shared__ double sA[32][33];
    __shared__ double sB[32][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
    const long long m0 = (long long)blockIdx.y * 32;
    const int n0 = blockIdx.x * 32;
    double acc[4] = {0, 0, 0, 0};
    for (int k0 = 0; k0 < K; k0 += 32) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int r = ty + q * 8;  // tile row index
            // sA[r][tx] = op(A)[m0 + r][k0 + tx]
            {
                const long long mi = m0 + (AT ? tx : r);
                const int ki = k0 + (AT ? r : tx);
                double v = 0.0;
                if (mi < M && ki < K) v = AT ? A[(long long)ki * lda + mi] : A[mi * lda + ki];
                if (AT) sA[tx][r] = v; else sA[r][tx] = v;
            }
            // sB[r][tx] = op(B)[k0 + r][n0 + tx]
            {
                const int ki = k0 + (BT ? tx : r);
                const int ni = n0 + (BT ? r : tx);
                double v = 0.0;
                if (ki < K && ni < N) v = BT ? B[(long long)ni * ldb + ki] : B[(long long)ki * ldb + ni];
                if (BT) sB[tx][r] = v; else sB[r][tx] = v;
            }
        }
        __syncthreads();
#pragma unroll 8
        for (int kk = 0; kk < 32; ++kk) {
            const double b = sB[kk][tx];
#pragma unroll
            for (int q = 0; q < 4; ++q) acc[q] = fma(sA[ty + q * 8][kk], b, acc[q]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const long long mi = m0 + ty + q * 8;
        const int ni = n0 + tx;
        if (mi < M && ni < N) {
            double v = alpha * acc[q];
            double* cp = C + mi * ldc + ni;
            if (beta != 0.0) v = fma(beta, *cp, v);
            *cp = v;
        }
    }
}

template <bool AT, bool BT>
int launch_generic(Ctx* c, long long M, int N, int K, double alpha, const double* A, int lda, const double* B, int ldb,
                   double beta, double* C, int ldc) {
    // one 32-row tile per blockIdx.y (<= 65535): a taller product -- gemm's 2^21-row chunks are 65536 tiles -- is launched
    // in row slices; every output row is computed the same way in either case
    constexpr long long MAX_ROWS = 65535LL * 32;
    for (long long r = 0; r < M; r += MAX_ROWS) {
        const long long mr = std::min(MAX_ROWS, M - r);
        const double* Ar = AT ? A + r : A + r * (long long)lda;
        dim3 grid((N + 31) / 32, (unsigned)((mr + 31) / 32));
        LQ_TRY((launch<gemm_generic_kernel<AT, BT>>(c, grid, 256, 0, c->stream, 0, Ar, B, C + r * (long long)ldc, mr, N, K, lda,
                                                    ldb, ldc, alpha, beta)));
    }
    return LQ_OK;
}

// when `parts` is given, the split-K partial sums are left in a workspace for a fused consumer kernel
struct Partials {
    DevBuf ws;
    double* ext = nullptr;       // caller-owned workspace (used instead of `ws` when large enough)
    size_t ext_bytes = 0;
    double* ptr = nullptr;       // where the partial sums are
    int splits = 1;
    long long stride = 0;
};
template <bool AT, bool BT>
int launch_fast(Ctx* c, long long M, int N, int Kmain, double alpha, const double* A, int lda, const double* B, int ldb,
                double beta, double* C, int ldc, Partials* parts = nullptr) {
    const bool skinny = AT && !BT && (M <= 64 || N <= 96);
    const long long tm = (M + BM - 1) / BM;
    const int tn = (N + BN - 1) / BN;
    const int KT = Kmain / BK;
    int splits = 1;
    const long long tiles = tm * tn;
    if (tiles < 2LL * c->sm_count && KT >= 16) {
        // split K so that tiles * splits fills whole waves of SMs (one CTA per SM): pick the split count in
        // [1, KT/8] with the best wave efficiency, preferring fewer splits (less workspace traffic) on ties
        const int max_splits = (int)std::min<long long>(std::max(1, KT / 8), (4LL * c->sm_count + tiles - 1) / tiles);
        double best_eff = 0.0;
        for (int sp = 1; sp <= max_splits; ++sp) {
            const long long ctas = tiles * sp;
            const long long waves = (ctas + c->sm_count - 1) / c->sm_count;
            // cost model: waves * (k-tiles per CTA + fixed per-CTA overhead of ~6 k-tiles)
            const double per = (double)((KT + sp - 1) / sp) + 6.0;
            const double eff = 1.0 / (waves * per);
            if (eff > best_eff * 1.02) {
                best_eff = eff;
                splits = sp;
            }
        }
    }
    GemmArgs g;
    g.A = A; g.B = B; g.M = M; g.N = N; g.K = Kmain; g.lda = lda; g.ldb = ldb;
    g.alpha = alpha; g.beta = beta; g.splits = splits;
    DevBuf ws_local;
    DevBuf& ws = parts ? parts->ws : ws_local;
    if (splits == 1 && !parts) {
        g.C = C; g.ldc = ldc; g.split_stride = 0;
    } else {
        const size_t need = (size_t)splits * M * N * sizeof(double);
        if (parts && parts->ext && parts->ext_bytes >= need) {
            g.C = parts->ext;
        } else {
            LQ_TRY(ws.alloc(c, need));
            g.C = ws.as<double>();
        }
        g.ldc = N; g.split_stride = M * (long long)N;
        if (parts) parts->ptr = g.C;
        if (splits == 1) { g.alpha = 1.0; g.beta = 0.0; }  // raw product into the workspace
    }
    CUtensorMap mapA, mapB;
    memset(&mapA, 0, sizeof(mapA));
    memset(&mapB, 0, sizeof(mapB));
    if (!AT) LQ_TRY(make_kmajor_map(c, &mapA, A, M, Kmain, lda));   // A stored M x K
    if (BT) LQ_TRY(make_kmajor_map(c, &mapB, B, N, Kmain, ldb));    // B stored N x K
    dim3 grid(tn, (unsigned)tm, splits);
    if (skinny)
        LQ_TRY((launch<gemm_dmma_kernel<AT, BT, AT && !BT>>(c, grid, GEMM_THREADS, GEMM_SMEM, c->stream, (int)GEMM_SMEM, g, mapA,
                                                            mapB)));
    else
        LQ_TRY((launch<gemm_dmma_kernel<AT, BT, false>>(c, grid, GEMM_THREADS, GEMM_SMEM, c->stream, (int)GEMM_SMEM, g, mapA, mapB)));
    if (parts) {
        parts->splits = splits;
        parts->stride = g.split_stride;
        return LQ_OK;
    }
    if (splits > 1) {
        const long long total = M * N;
        const int blocks = (int)std::min<long long>((total + 255) / 256, (long long)c->sm_count * 8);
        return launch<splitk_reduce_kernel>(c, blocks, 256, 0, c->stream, 0, g.C, splits, g.split_stride, M, N, alpha, beta, C,
                                            ldc);
    }
    return LQ_OK;
}

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// W2 (kb x nc) = op(T) * (sum_z P_z),  P_z (kb x nc) the split-K partials of V^T C;  kb <= 128.
// CTA b owns 32 columns.  op(T) is staged in shared memory as Ts[k][i] = op(T)[i][k], the summed partials as
// Ws[k][c]; thread (c = tid & 31, row group tid >> 5) forms 4 outputs at a time so that every Ws load feeds 4 FMAs.
__global__ void __launch_bounds__(1024) reduce_apply_t_kernel(const double* __restrict__ P, int splits, long long stride,
                                                             int kb, int nc, const double* __restrict__ T, int ldt,
                                                             int trans_t, double* __restrict__ W2) {
    extern __shared__ double sh_rat[];
    const int pt = kb + 1;
    double* Ts = sh_rat;                 // [kb][kb + 1]
    double* Ws = sh_rat + kb * pt;       // [kb][33]
    const int c0 = blockIdx.x * 32;
    const int ncv = min(32, nc - c0);
    const int NT = blockDim.x;  // 1024
    // stage op(T): 4 independent global loads in flight per thread
    for (int e0 = threadIdx.x; e0 < kb * kb; e0 += NT * 4) {
        double v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int e = e0 + u * NT;
            const int r = e / kb, q = e - r * kb;
            v[u] = (e < kb * kb && q >= r) ? T[(long long)r * ldt + q] : 0.0;  // T is upper triangular
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int e = e0 + u * NT;
            if (e < kb * kb) {
                const int r = e / kb, q = e - r * kb;
                if (trans_t) Ts[r * pt + q] = v[u];   // op(T)[i][k] = T[k][i]  ->  Ts[k = r][i = q]
                else Ts[q * pt + r] = v[u];           // op(T)[i][k] = T[i][k]  ->  Ts[k = q][i = r]
            }
        }
    }
    // sum the split-K partials of my 32 columns: thread (k = tid >> 5 (+32, ...), cc = tid & 31), 8 splits in flight
    {
        const int cc = threadIdx.x & 31;
        const bool ok = cc < ncv;
        for (int k = threadIdx.x >> 5; k < kb; k += NT / 32) {
            double sa[8] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
            const double* src = P + (long long)k * nc + c0 + cc;
            if (ok) {
                int z = 0;
                for (; z + 8 <= splits; z += 8) {
#pragma unroll
                    for (int u = 0; u < 8; ++u) sa[u] += src[(z + u) * stride];
                }
                for (; z < splits; ++z) sa[0] += src[z * stride];
            }
            Ws[k * 33 + cc] = ((sa[0] + sa[1]) + (sa[2] + sa[3])) + ((sa[4] + sa[5]) + (sa[6] + sa[7]));
        }
    }
    __syncthreads();
    const int cc = threadIdx.x & 31;
    for (int i0 = (threadIdx.x >> 5) * 4; i0 < kb; i0 += NT / 8) {
        double acc[4] = {0.0, 0.0, 0.0, 0.0};
        // op(T)[i][k] != 0 only for k <= i (transpose) or k >= i (no transpose)
        const int klo = trans_t ? 0 : i0;
        const int khi = trans_t ? min(kb, i0 + 4) : kb;
        for (int k = klo; k < khi; ++k) {
            const double w = Ws[k * 33 + cc];
#pragma unroll
            for (int r = 0; r < 4; ++r) acc[r] = fma(Ts[k * pt + i0 + r], w, acc[r]);
        }
        if (cc < ncv) {
#pragma unroll
            for (int r = 0; r < 4; ++r)
                if (i0 + r < kb) W2[(long long)(i0 + r) * nc + c0 + cc] = acc[r];
        }
    }
}

}  // namespace

// ------------------------------------------------------------------ rank-K products (K <= 128) with one operand resident
// C = alpha * A * B + beta * C  (NN) where the contraction is short (the 128 reflectors of a block update
// C -= V W, or U = A (V S^-1), Q = A R^-1 on tall-skinny matrices).  With K = 128 a 128 x 128 output tile has only
// 8 k-tiles, so the generic kernel spends a third of each CTA's life filling its pipeline and reading C.  Here a
// persistent CTA keeps the B column tile (K x 128) resident in shared memory for its whole life and walks down the
// A / C row tiles (tall-skinny products).  The producer warp runs ahead across tile boundaries, so the next tile's
// operands land during the current epilogue.
constexpr int RK_KT_MAX = 8;  // K <= 128
constexpr size_t RK_SMEM_BSTAT = (size_t)RK_KT_MAX * TILE_BYTES + (size_t)STAGES * BM * BK * 8 + 16 * sizeof(uint64_t) + 1024;

struct RankArgs {
    const double* B;
    double* C;
    long long M;
    int N, K;
    int ldb, ldc;
    double alpha, beta;
};

__global__ void __launch_bounds__(GEMM_THREADS, 1) gemm_rank_kernel(const RankArgs g, const __grid_constant__ CUtensorMap mapA) {
    extern __shared__ unsigned char smem_dyn[];
    unsigned char* smem_raw = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
    constexpr int ABOX = BM * BK;  // doubles per swizzled A box
    // layout: [resident B tile][streamed A ring][barriers]
    double* res = reinterpret_cast<double*>(smem_raw);
    double* ring = res + RK_KT_MAX * TILE_DOUBLES;
    uint64_t* bars = reinterpret_cast<uint64_t*>(ring + STAGES * ABOX);
    uint64_t* full = bars;
    uint64_t* empty = bars + STAGES;
    uint64_t* res_full = bars + 2 * STAGES;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int KT = g.K / BK;
    const long long tm = (g.M + BM - 1) / BM;
    // fixed column tile (resident B) and walk over the row tiles (streamed A)
    const long long fix = blockIdx.x;
    const long long walk0 = blockIdx.y;
    const long long walk_step = gridDim.y;

    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], 8);
        }
        mbar_init(res_full, 1);
        mbar_fence_init();
    }
    __syncthreads();

    if (warp == 8) {
        // ===================== producer =====================
        const int n0 = (int)fix * BN;
        const int nvalid = min(BN, g.N - n0);
        if (lane == 0) mbar_expect_tx(res_full, (uint32_t)(KT * BK * nvalid * 8));
        __syncwarp();
        if (lane < BK)
            for (int kt = 0; kt < KT; ++kt)
                bulk_g2s(res + kt * TILE_DOUBLES + lane * PM, g.B + (long long)(kt * BK + lane) * g.ldb + n0, nvalid * 8, res_full);
        int it = 0;
        for (long long w = walk0; w < tm; w += walk_step) {
            for (int kt = 0; kt < KT; ++kt, ++it) {
                const int s = it % STAGES;
                const uint32_t ph = (it / STAGES) & 1;
                mbar_wait(&empty[s], ph ^ 1);
                if (lane == 0) {
                    mbar_expect_tx(&full[s], (uint32_t)(ABOX * 8));
                    tma_load_2d(ring + s * ABOX, &mapA, kt * BK, (int)(w * BM), &full[s]);
                }
            }
        }
        return;
    }

    // ===================== consumers =====================
    const int wm = warp >> 2, wn = warp & 3;
    const int gq = lane >> 2, tq = lane & 3;
    mbar_wait(res_full, 0);
    int it = 0;
    for (long long w = walk0; w < tm; w += walk_step) {
        const long long m0 = w * BM;
        const int n0 = (int)fix * BN;
        const int mvalid = (int)min((long long)BM, g.M - m0);
        const int nvalid = min(BN, g.N - n0);
        if (g.beta != 0.0 && g.beta != 1.0 && tq == 0) {
            // pull my part of the C tile into L2 while the 8 k-tiles run
#pragma unroll
            for (int h = 0; h < 8; ++h) {
                const int r = wm * 64 + (h >> 1) * 16 + gq + (h & 1) * 8;
                if (r < mvalid) {
                    const double* crow = g.C + (m0 + r) * (long long)g.ldc + n0 + wn * 32;
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(crow));
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(crow + 16));
                }
            }
        }
        double acc[4][4][4];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
                for (int e = 0; e < 4; ++e) acc[i][j][e] = 0.0;
        for (int kt = 0; kt < KT; ++kt, ++it) {
            const int s = it % STAGES;
            const uint32_t ph = (it / STAGES) & 1;
            mbar_wait(&full[s], ph);
            const double* sA = ring + s * ABOX;
            const double* sB = res + kt * TILE_DOUBLES;
#pragma unroll
            for (int ks = 0; ks < BK / 8; ++ks) {
                double bf[4][2];
                const int kA = ks * 8 + tq;
#pragma unroll
                for (int jn = 0; jn < 4; ++jn) {
                    const int c = wn * 32 + jn * 8 + gq;
                    bf[jn][0] = sB[kA * PM + c];
                    bf[jn][1] = sB[(kA + 4) * PM + c];
                }
#pragma unroll
                for (int im = 0; im < 4; ++im) {
                    double af[4];
                    const int r = wm * 64 + im * 16 + gq;
                    af[0] = sA[sw_idx(r, gq, kA)];
                    af[1] = sA[sw_idx(r + 8, gq, kA)];
                    af[2] = sA[sw_idx(r, gq, kA + 4)];
                    af[3] = sA[sw_idx(r + 8, gq, kA + 4)];
#pragma unroll
                    for (int jn = 0; jn < 4; ++jn) dmma_16x8x8(acc[im][jn], af, bf[jn]);
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[s]);
        }
        // ---- epilogue of this tile
        const bool vec2 = ((g.ldc & 1) == 0) && ((reinterpret_cast<uintptr_t>(g.C) & 15) == 0);
#pragma unroll
        for (int im = 0; im < 4; ++im) {
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const int r = wm * 64 + im * 16 + gq + half * 8;
                if (r >= mvalid) continue;
                double* crow = g.C + (m0 + r) * (long long)g.ldc + n0;
                if (g.beta == 1.0) {
#pragma unroll
                    for (int jn = 0; jn < 4; ++jn) {
                        const int c = wn * 32 + jn * 8 + 2 * tq;
                        if (c < nvalid) red_add(crow + c, g.alpha * acc[im][jn][half * 2 + 0]);
                        if (c + 1 < nvalid) red_add(crow + c + 1, g.alpha * acc[im][jn][half * 2 + 1]);
                    }
                    continue;
                }
                double cold[4][2];
                if (g.beta != 0.0) {
#pragma unroll
                    for (int jn = 0; jn < 4; ++jn) {
                        const int c = wn * 32 + jn * 8 + 2 * tq;
                        cold[jn][0] = 0.0;
                        cold[jn][1] = 0.0;
                        if (vec2 && c + 1 < nvalid) {
                            const double2 t2 = *reinterpret_cast<const double2*>(crow + c);
                            cold[jn][0] = t2.x;
                            cold[jn][1] = t2.y;
                        } else {
                            if (c < nvalid) cold[jn][0] = crow[c];
                            if (c + 1 < nvalid) cold[jn][1] = crow[c + 1];
                        }
                    }
                }
#pragma unroll
                for (int jn = 0; jn < 4; ++jn) {
                    const int c = wn * 32 + jn * 8 + 2 * tq;
                    double v0 = g.alpha * acc[im][jn][half * 2 + 0];
                    double v1 = g.alpha * acc[im][jn][half * 2 + 1];
                    if (g.beta != 0.0) {
                        v0 = fma(g.beta, cold[jn][0], v0);
                        v1 = fma(g.beta, cold[jn][1], v1);
                    }
                    if (vec2 && c + 1 < nvalid) {
                        *reinterpret_cast<double2*>(crow + c) = make_double2(v0, v1);
                    } else {
                        if (c < nvalid) crow[c] = v0;
                        if (c + 1 < nvalid) crow[c + 1] = v1;
                    }
                }
            }
        }
    }
}

// returns LQ_ERR_UNSUPPORTED when the shape is not a rank-K product this kernel takes
int gemm_rank(Ctx* c, long long M, int N, int K, double alpha, const double* A, int lda, const double* B, int ldb, double beta,
              double* C, int ldc) {
    if (K > RK_KT_MAX * BK || K % BK != 0 || K < BK || (N % 2) != 0 || M < 2 * BM) return LQ_ERR_UNSUPPORTED;
    const long long tm = (M + BM - 1) / BM;
    const int tn = (N + BN - 1) / BN;
    // measured on B200: the B-stationary walk wins on tall-skinny products (30.2 vs 27.8 TFLOP/s at 2^20 x 128 x 128).
    // Wide outputs (4+ column tiles) and short ones stay on the generic kernel: an A-stationary walk for square block
    // updates did not beat it (23.6 vs 25.0).
    if (tn >= 4 || tm < 4) return LQ_ERR_UNSUPPORTED;
    CUtensorMap mapA;
    LQ_TRY(make_kmajor_map(c, &mapA, A, M, K, lda));
    RankArgs g;
    g.B = B; g.C = C; g.M = M; g.N = N; g.K = K; g.ldb = ldb; g.ldc = ldc; g.alpha = alpha; g.beta = beta;
    // CTAs per column tile: fill the SMs once (persistent), at most one CTA per row tile
    long long per_fixed = std::max<long long>(1, std::min<long long>(tm, (c->sm_count + tn - 1) / tn));
    // prefer a whole number of equal walks
    while (per_fixed > 1 && tn * per_fixed > (long long)c->sm_count && tn * (per_fixed - 1) >= c->sm_count * 3 / 4)
        --per_fixed;
    dim3 grid((unsigned)tn, (unsigned)per_fixed);
    return launch<gemm_rank_kernel>(c, grid, GEMM_THREADS, RK_SMEM_BSTAT, c->stream, (int)RK_SMEM_BSTAT, g, mapA);
}


// ------------------------------------------------------------------ rank-K update  C += alpha * A * B   (NN, small K)
// The block-reflector applications of the blocked QR end in C -= V W with K = 128: a 128 x 128 tile spends as long in
// its prologue (first TMA round trip) and epilogue as in 3 of its 8 k-tiles, and one CTA per SM cannot hide either
// (DMMA pipe 70 %).  This kernel halves the tile (128 x 64: 64 accumulator registers, a 100 KB operand ring), so TWO
// CTAs share an SM and one CTA's prologue / epilogue runs under the other's main loop.  Same ingredients as
// gemm_dmma_kernel: K-major A tiles as one swizzled 2-D TMA box per stage, B rows as bulk copies, mma.sync m16n8k8.f64,
// the result leaves through the TMA engine as one bulk reduce-add per row (no read-back of C, one writer per element).
constexpr int UBN = 64;
constexpr int UPB = UBN + 4;                 // pitch of a [k][n] B tile
constexpr int U_STAGES = 4;
constexpr int U_STAGE_BYTES = 25600;         // 16 KiB A box + 16 x 68 doubles of B, rounded to 1 KiB (swizzle alignment)
constexpr int U_EPI_PITCH = UBN + 8;         // staged C row (a quarter-warp's 16-byte stores hit distinct banks)
constexpr size_t UPD_SMEM = (size_t)U_STAGES * U_STAGE_BYTES + 2 * U_STAGES * sizeof(uint64_t) + 1024;
static_assert(BM * BK * 8 + BK * UPB * 8 <= U_STAGE_BYTES, "stage holds an A box and a B tile");
static_assert((size_t)BM * U_EPI_PITCH * 8 <= (size_t)U_STAGES * U_STAGE_BYTES, "the staged C tile reuses the operand ring");

struct UpdArgs {
    const double* B;
    double* C;
    long long M;
    int N, K;
    int ldb, ldc;
    double alpha;
    int overwrite;  // 0: C += alpha A B (bulk reduce-add), 1: C = alpha A B (bulk store)
};

__global__ void __launch_bounds__(GEMM_THREADS, 2) gemm_upd_kernel(const UpdArgs g, const __grid_constant__ CUtensorMap mapA) {
    extern __shared__ unsigned char smem_dyn[];
    unsigned char* smem_raw = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + (size_t)U_STAGES * U_STAGE_BYTES);
    uint64_t* empty = full + U_STAGES;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long m0 = (long long)blockIdx.y * BM;
    const int n0 = blockIdx.x * UBN;
    const int mvalid = (int)min((long long)BM, g.M - m0);
    const int nvalid = min(UBN, g.N - n0);
    const int nkt = g.K / BK;

    if (threadIdx.x == 0) {
        for (int s = 0; s < U_STAGES; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], 8);
        }
        mbar_fence_init();
    }
    __syncthreads();

    if (warp == 8) {
        // ===================== producer =====================
        const uint32_t bytes = (uint32_t)(BM * BK * 8) + (uint32_t)(BK * nvalid * 8);
        for (int it = 0; it < nkt; ++it) {
            const int s = it % U_STAGES;
            const uint32_t ph = (it / U_STAGES) & 1;
            mbar_wait(&empty[s], ph ^ 1);
            double* sA = reinterpret_cast<double*>(smem_raw + (size_t)s * U_STAGE_BYTES);
            double* sB = sA + BM * BK;
            const int k0 = it * BK;
            if (lane == 0) mbar_expect_tx(&full[s], bytes);
            __syncwarp();
            if (lane == 0) tma_load_2d(sA, &mapA, k0, (int)m0, &full[s]);
            if (lane >= 16) {
                const int kk = lane - 16;
                bulk_g2s(sB + kk * UPB, g.B + (long long)(k0 + kk) * g.ldb + n0, nvalid * 8, &full[s]);
            }
        }
        return;
    }

    // ===================== consumers: 4 (m) x 2 (n) warps, 32 x 32 each =====================
    const int wm = warp >> 1, wn = warp & 1;
    const int gq = lane >> 2, tq = lane & 3;
    double acc[2][4][4];
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j)
#pragma unroll
            for (int e = 0; e < 4; ++e) acc[i][j][e] = 0.0;

    for (int it = 0; it < nkt; ++it) {
        const int s = it % U_STAGES;
        const uint32_t ph = (it / U_STAGES) & 1;
        mbar_wait(&full[s], ph);
        const double* sA = reinterpret_cast<const double*>(smem_raw + (size_t)s * U_STAGE_BYTES);
        const double* sB = sA + BM * BK;
#pragma unroll
        for (int ks = 0; ks < BK / 8; ++ks) {
            const int kA = ks * 8 + tq;
            double bf[4][2];
#pragma unroll
            for (int jn = 0; jn < 4; ++jn) {
                const int c = wn * 32 + jn * 8 + gq;
                bf[jn][0] = sB[kA * UPB + c];
                bf[jn][1] = sB[(kA + 4) * UPB + c];
            }
#pragma unroll
            for (int im = 0; im < 2; ++im) {
                double af[4];
                const int r = wm * 32 + im * 16 + gq;
                af[0] = sA[sw_idx(r, gq, kA)];
                af[1] = sA[sw_idx(r + 8, gq, kA)];
                af[2] = sA[sw_idx(r, gq, kA + 4)];
                af[3] = sA[sw_idx(r + 8, gq, kA + 4)];
#pragma unroll
                for (int jn = 0; jn < 4; ++jn) dmma_16x8x8(acc[im][jn], af, bf[jn]);
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[s]);
    }

    // ===================== epilogue: stage the tile, one bulk reduce-add per row =====================
    consumer_bar_sync();  // every consumer warp is done reading the operand stages
    double* stg = reinterpret_cast<double*>(smem_raw);
#pragma unroll
    for (int im = 0; im < 2; ++im)
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const int r = wm * 32 + im * 16 + gq + half * 8;
#pragma unroll
            for (int jn = 0; jn < 4; ++jn) {
                const int c = wn * 32 + jn * 8 + 2 * tq;
                *reinterpret_cast<double2*>(stg + r * U_EPI_PITCH + c) =
                    make_double2(g.alpha * acc[im][jn][half * 2 + 0], g.alpha * acc[im][jn][half * 2 + 1]);
            }
        }
    fence_proxy_async();
    consumer_bar_sync();
    if (lane < 16) {
        const int r = warp * 16 + lane;
        if (r < mvalid) {
            double* dst = g.C + (m0 + r) * (long long)g.ldc + n0;
            if (g.overwrite) bulk_s2g(dst, stg + r * U_EPI_PITCH, (uint32_t)nvalid * 8u);
            else bulk_red_add_f64(dst, stg + r * U_EPI_PITCH, (uint32_t)nvalid * 8u);
        }
    }
    bulk_commit();
    bulk_wait_read<0>();
}

// C (+)= alpha * A * B for row-major A (M x K, lda), B (K x N, ldb), K a small multiple of 16; LQ_ERR_UNSUPPORTED otherwise
int gemm_update(Ctx* c, long long M, int N, int K, double alpha, const double* A, int lda, const double* B, int ldb, double* C,
                int ldc, bool overwrite) {
    if (K % BK != 0 || K < BK || K > 512 || (N % 2) != 0 || (ldc % 2) != 0 || !aligned16(C) || M < BM || N < UBN)
        return LQ_ERR_UNSUPPORTED;
    const long long tm = (M + BM - 1) / BM;
    const int tn = (N + UBN - 1) / UBN;
    if (tm * tn < 2LL * c->sm_count) return LQ_ERR_UNSUPPORTED;  // small outputs: the split-K / one-tile paths
    CUtensorMap mapA;
    LQ_TRY(make_kmajor_map(c, &mapA, A, M, K, lda));
    UpdArgs g;
    g.B = B; g.C = C; g.M = M; g.N = N; g.K = K; g.ldb = ldb; g.ldc = ldc; g.alpha = alpha; g.overwrite = overwrite ? 1 : 0;
    dim3 grid((unsigned)tn, (unsigned)tm);
    return launch<gemm_upd_kernel>(c, grid, GEMM_THREADS, UPD_SMEM, c->stream, (int)UPD_SMEM, g, mapA);
}

int gemm(Ctx* c, bool ta, bool tb, long long M, int N, int K, double alpha, const double* A, int lda, const double* B,
         int ldb, double beta, double* C, int ldc) {
    if (M <= 0 || N <= 0) return LQ_OK;
    // the kernels index the row tiles with blockIdx.y (<= 65535): very tall products (2^23 x 128 on one GPU) go in row chunks
    constexpr long long ROW_CHUNK = 1LL << 21;  // 16384 tiles of 128 rows (launch_generic slices its 32-row tiles further)
    if (M > ROW_CHUNK) {
        for (long long r = 0; r < M; r += ROW_CHUNK) {
            const long long mc = std::min(ROW_CHUNK, M - r);
            const double* Ar = ta ? A + r : A + r * (long long)lda;  // op(A) row r: column r of a transposed A
            LQ_TRY(gemm(c, ta, tb, mc, N, K, alpha, Ar, lda, B, ldb, beta, C + r * (long long)ldc, ldc));
        }
        return LQ_OK;
    }
    if (K <= 0) {
        // C = beta * C
        if (beta == 1.0) return LQ_OK;
        return ta ? launch_generic<true, false>(c, M, N, 0, alpha, A, lda, B, ldb, beta, C, ldc)
                  : launch_generic<false, false>(c, M, N, 0, alpha, A, lda, B, ldb, beta, C, ldc);
    }
    const int Kmain = K - K % BK;
    bool fast = Kmain >= BK && aligned16(A) && aligned16(B) && (lda % 2 == 0) && (ldb % 2 == 0) && (M * (long long)N >= 32 * 32);
    if (ta) fast = fast && (M % 2 == 0);   // M-major rows copied in whole 16-byte units
    if (!tb) fast = fast && (N % 2 == 0);
    if (!fast) {
        if (ta && tb) return launch_generic<true, true>(c, M, N, K, alpha, A, lda, B, ldb, beta, C, ldc);
        if (ta) return launch_generic<true, false>(c, M, N, K, alpha, A, lda, B, ldb, beta, C, ldc);
        if (tb) return launch_generic<false, true>(c, M, N, K, alpha, A, lda, B, ldb, beta, C, ldc);
        return launch_generic<false, false>(c, M, N, K, alpha, A, lda, B, ldb, beta, C, ldc);
    }
    int rc;
    if (!ta && !tb && Kmain == K) {
        // small K: the two-CTAs-per-SM kernel (in-place accumulation or plain product), then the B-stationary walk
        if (beta == 1.0 || beta == 0.0) {
            rc = gemm_update(c, M, N, K, alpha, A, lda, B, ldb, C, ldc, beta == 0.0);
            if (rc != LQ_ERR_UNSUPPORTED) return rc;
        }
        rc = gemm_rank(c, M, N, K, alpha, A, lda, B, ldb, beta, C, ldc);
        if (rc != LQ_ERR_UNSUPPORTED) return rc;
    }
    if (ta && tb) rc = launch_fast<true, true>(c, M, N, Kmain, alpha, A, lda, B, ldb, beta, C, ldc);
    else if (ta) rc = launch_fast<true, false>(c, M, N, Kmain, alpha, A, lda, B, ldb, beta, C, ldc);
    else if (tb) rc = launch_fast<false, true>(c, M, N, Kmain, alpha, A, lda, B, ldb, beta, C, ldc);
    else rc = launch_fast<false, false>(c, M, N, Kmain, alpha, A, lda, B, ldb, beta, C, ldc);
    if (rc != LQ_OK) return rc;
    if (Kmain < K) {
        // K remainder: C += alpha * op(A)[:, Kmain:] * op(B)[Kmain:, :]
        const double* A2 = ta ? A + (long long)Kmain * lda : A + Kmain;
        const double* B2 = tb ? B + Kmain : B + (long long)Kmain * ldb;
        const int Kr = K - Kmain;
        if (ta && tb) return launch_generic<true, true>(c, M, N, Kr, alpha, A2, lda, B2, ldb, 1.0, C, ldc);
        if (ta) return launch_generic<true, false>(c, M, N, Kr, alpha, A2, lda, B2, ldb, 1.0, C, ldc);
        if (tb) return launch_generic<false, true>(c, M, N, Kr, alpha, A2, lda, B2, ldb, 1.0, C, ldc);
        return launch_generic<false, false>(c, M, N, Kr, alpha, A2, lda, B2, ldb, 1.0, C, ldc);
    }
    return LQ_OK;
}

int vtc_finish(Ctx* c, const double* partials, int splits, long long stride, int kb, int nc, const double* T, int ldt,
               bool trans_t, double* W2);

// W2 (kb x nc, ld nc) = op(T) * (V^T C):  V (mk x kb, ldv), C (mk x nc, ldc), T (kb x kb upper, ldt), kb <= 128.
// One split-K tensor-core GEMM whose partial sums feed a fused reduce + triangular-multiply kernel.
int gemm_vtc_apply_t(Ctx* c, int kb, int nc, int mk, const double* V, int ldv, const double* Cm, int ldc, const double* T,
                     int ldt, bool trans_t, double* W2) {
    if (kb <= 0 || nc <= 0) return LQ_OK;
    const int Kmain = mk - mk % BK;
    const bool fast = kb <= 128 && Kmain >= BK && Kmain == mk && aligned16(V) && aligned16(Cm) && (ldv % 2 == 0) &&
                      (ldc % 2 == 0) && (kb % 4 == 0) && (nc % 2 == 0);
    if (!fast) {
        DevBuf W;
        LQ_TRY(W.alloc(c, sizeof(double) * (size_t)kb * nc));
        LQ_TRY(gemm(c, true, false, kb, nc, mk, 1.0, V, ldv, Cm, ldc, 0.0, W.as<double>(), nc));
        return gemm(c, trans_t, false, kb, nc, kb, 1.0, T, ldt, W.as<double>(), nc, 0.0, W2, nc);
    }
    Partials parts;
    LQ_TRY((launch_fast<true, false>(c, kb, nc, Kmain, 1.0, V, ldv, Cm, ldc, 0.0, nullptr, nc, &parts)));
    return vtc_finish(c, parts.ptr, parts.splits, parts.stride, kb, nc, T, ldt, trans_t, W2);
}

int vtc_finish(Ctx* c, const double* partials, int splits, long long stride, int kb, int nc, const double* T, int ldt,
               bool trans_t, double* W2) {
    // opted in once to the 128-column maximum, whatever kb the first call has
    const size_t rat_smem = ((size_t)kb * (kb + 1) + (size_t)kb * 33 + 8) * sizeof(double);
    return launch<reduce_apply_t_kernel>(c, (nc + 31) / 32, 1024, rat_smem, c->stream,
                                         (int)((128 * 129 + 128 * 33 + 8) * sizeof(double)), partials, splits, stride, kb, nc, T,
                                         ldt, trans_t ? 1 : 0, W2);
}

}  // namespace lq

using namespace lq;
extern "C" int lq_gemm_dev(lq_ctx* h, int transa, int transb, int64_t m, int n, int k, double alpha, const double* A,
                           int lda, const double* B, int ldb, double beta, double* C, int ldc) {
    Ctx* c = as_ctx(h);
    if (!c) return LQ_ERR_ARG;
    LQ_CUDA(c, cudaSetDevice(c->device));
    return gemm(c, transa != 0, transb != 0, m, n, k, alpha, A, lda, B, ldb, beta, C, ldc);
}

// Internal (device-pointer) operations shared between the translation units.
#pragma once

#include <algorithm>
#include <atomic>

#include "ctx.cuh"

namespace lq {

// CTAs of a grid-stride element-wise kernel over `total` elements: one element per thread, at most 8 CTAs of 256 per SM
inline int grid_for(Ctx* c, long long total) {
    return (int)std::max<long long>(1, std::min<long long>((total + 255) / 256, (long long)c->sm_count * 8));
}

// ---- gemm.cu: row-major C = alpha * op(A) * op(B) + beta * C on the context stream.
// FP64 tensor-core (DMMA) kernel fed by bulk-async (TMA engine) copies when shapes are aligned,
// plain tiled kernel otherwise.
int gemm(Ctx* c, bool transa, bool transb, long long m, int n, int k, double alpha, const double* A, int lda,
         const double* B, int ldb, double beta, double* C, int ldc);

// W2 (kb x nc) = op(T) (V^T C): split-K GEMM + fused reduce / triangular multiply (block-reflector applications)
int gemm_vtc_apply_t(Ctx* c, int kb, int nc, int mk, const double* V, int ldv, const double* Cm, int ldc, const double* T,
                     int ldt, bool trans_t, double* W2);

// second phase of the above (reduction of the split-K partial sums + op(T)), used by gemm_vtc_apply_t
int vtc_finish(Ctx* c, const double* partials, int splits, long long stride, int kb, int nc, const double* T, int ldt,
               bool trans_t, double* W2);

// ---- blocked_qr.cu: single-matrix blocked compact-WY Householder (linalg/qr.py:52-100)
int blocked_householder_qr(Ctx* c, const double* A, int m, int n, double* Q, double* R);
// factor only: A (m x n, lda) overwritten by R (upper) ; V (m x n, ldv) receives unit-norm reflectors
// (zeros above the diagonal), skipped reflectors are zero columns.  Optional B (m x nrhs) gets Q^T B.
int blocked_householder_factor(Ctx* c, double* A, int lda, int m, int n, double* V, int ldv, double* B, int ldb,
                               int nrhs);
// info (device, may be null): 0, or 1 + the first column whose R[j][j] is exactly 0 (the solve is singular)
int large_lstsq_householder(Ctx* c, const double* A, const double* B, int m, int n, int nrhs, double* X, int* info);
// dst (rows x cols_dst, ldd) = [src | 0] (src rows x cols_src, lds)
int pad_columns(Ctx* c, const double* src, int lds, double* dst, int ldd, long long rows, int cols_src, int cols_dst);
// R X = Y in place, one thread per right-hand side (R n x n upper triangular, ldr; Y n x k, ldy)
int backsub_per_column(Ctx* c, const double* R, int ldr, double* Y, int ldy, int n, int k);
// Largest cluster of the barrier.cluster panel kernel the device holds (16, 8, 4, 2 or 1) -> c->max_cluster.  One
// occupancy query when the context is created; launches nothing.
int measure_max_cluster(Ctx* c);

// ---- large_mgs.cu: single-matrix MGS for shapes beyond one CTA's shared memory
int large_mgs_qr(Ctx* c, const double* A, int m, int n, int reorth, double* Q, double* R, int* info);
int large_lstsq_mgs(Ctx* c, const double* A, const double* B, int m, int n, int nrhs, double* X, int* info);

// ---- lstsq_stream.cu: K3 streaming Householder least squares (n <= 64, nrhs <= 32).  info (may be null): per system 0,
// or 1 + the first column whose R[j][j] is exactly 0.  LQ_ERR_UNSUPPORTED if the shape is not covered.
bool lstsq_stream_kernel_supported(int m, int n, int nrhs);
int lstsq_stream_kernel_launch(Ctx* c, cudaStream_t st, const double* A, const double* B, long long batch, int m,
                               int n, int nrhs, double* X, int* info);

// round 2: one warp per system, block reflectors on DMMA (n <= 64, nrhs <= 16).  info (may be null): per system, 0 or
// 1 + the first column with |R[j][j]| < 1e-12 (info_mode 1, the MGS test of linalg/qr.py:40-41) / == 0 (info_mode 2)
bool lstsq_tile_kernel_supported(int m, int n, int nrhs);
int lstsq_tile_kernel_launch(Ctx* c, cudaStream_t st, const double* A, const double* B, long long batch, int m, int n,
                             int nrhs, double* X, int* info, int info_mode);

// ---- syrk.cu: G (n x n, both triangles) = A^T A for n <= 128, upper-triangle blocks only; LQ_ERR_UNSUPPORTED otherwise
int syrk_tn(Ctx* c, const double* A, int lda, long long m, int n, double* G, int ldg);
// G (n x n, both triangles) = Q^T Q and C (n x nrhs) = Q^T B in one pass (Q m x n, B m x nrhs, densely packed).  Taken for
// even n <= 128, even nrhs <= 32, m >= 1024 and 16-byte aligned Q and B (syrk_strip_supported); LQ_ERR_UNSUPPORTED otherwise.
bool syrk_strip_supported(const double* Q, long long m, int n, const double* B, int nrhs);
int syrk_strip_tn(Ctx* c, const double* Q, long long m, int n, const double* B, int nrhs, double* G, double* C);

// G = A^T A (A m x n, row stride lda): the symmetric rank-k kernel when the shape allows, the general TN GEMM otherwise
inline int gram(Ctx* c, const double* A, int lda, long long m, int n, double* G) {
    const int rc = syrk_tn(c, A, lda, m, n, G, n);
    if (rc != LQ_ERR_UNSUPPORTED) return rc;
    return gemm(c, true, false, n, n, (int)m, 1.0, A, lda, A, lda, 0.0, G, n);
}

// ---- eigh_svd.cu: the Jacobi eigen-solver and the economy SVD through the Gram matrix
// psd: the caller guarantees a positive semi-definite G (a Gram matrix): a well-conditioned one then gets its eigenvectors as
// the normalised converged columns b_i = lambda_i v_i instead of replaying the rotation log
int eigh_jacobi(Ctx* c, const double* G, int n, double* lambda_desc, double* V, bool psd = false);
// rank_dev (device, may be null) receives the rank too, stream-ordered
int svd_gram_local(Ctx* c, const double* A, long long m, int n, double tol, double* U, double* s, double* Vt,
                   int* rank_host, bool sharded, int* rank_dev = nullptr);

// ---- tsqr.cu: thin QR and least squares of tall-skinny matrices, on one GPU or row-sharded
int tsqr_local(Ctx* c, const double* A, long long m, int n, double* Q, double* R, bool sharded);
// min ||A X - B|| for a tall-skinny A (m x n) and B (m x nrhs): CholeskyQR2 pipeline, Householder fallbacks.  info (device):
// 0, or 1 + the first column whose R[j][j] is exactly 0
int lstsq_tsqr_local(Ctx* c, const double* A, long long m, int n, const double* B, int nrhs, double* X, int* info, bool sharded);

// ---- batched dispatchers (api_batched.cu).  Each *_one_launch predicate says whether a shape takes one kernel launch
// for the whole batch, on any stream `st`.  Otherwise the dispatcher runs the single-matrix path matrix by matrix, and
// `st` must be the context stream.
// qr32: 32 x 32 matrices go to the batched 32 x 32 kernel; false keeps them on the one-CTA kernel (the single-matrix
// entry point)
bool hh_qr_batched_one_launch(Ctx* c, int m, int n);
int hh_qr_batched_stream(Ctx* c, cudaStream_t st, const double* A, long long batch, int m, int n, double* Q,
                         double* R, bool qr32);
// info (device, may be null): per matrix 0, or 1 + the first column with R[j][j] < 1e-12 (linalg/qr.py:40-41)
bool mgs_qr_batched_one_launch(Ctx* c, int m, int n);
int mgs_qr_batched_stream(Ctx* c, cudaStream_t st, const double* A, long long batch, int m, int n, int reorth,
                          double* Q, double* R, int* info);
// info (device, may be null): per system 0, or 1 + the first column whose R[j][j] is exactly 0
bool lstsq_hh_batched_one_launch(Ctx* c, int m, int n, int nrhs);
int lstsq_hh_batched_stream(Ctx* c, cudaStream_t st, const double* A, const double* B, long long batch, int m, int n,
                            int nrhs, double* X, int* info = nullptr);
bool lstsq_mgs_batched_one_launch(Ctx* c, int m, int n, int nrhs);
int lstsq_mgs_batched_stream(Ctx* c, cudaStream_t st, const double* A, const double* B, long long batch, int m, int n,
                             int nrhs, double* X, int* info);
// one launch when svd_small_supported(m, n) (batched_svd_small.cuh)
int svd_batched_stream(Ctx* c, cudaStream_t st, const double* A, long long batch, int m, int n, double tol, double* U,
                       double* s, double* Vt, int* rank);

// argument checks shared by the batched entry points (device and host pointers)
#define LQ_ARGS_QR(c, A, batch, m, n)                                                                       \
    LQ_REQUIRE(c, c != nullptr, LQ_ERR_ARG, "null context");                                               \
    LQ_REQUIRE(c, batch >= 0 && m >= 1 && n >= 1, LQ_ERR_SHAPE, "bad shape batch=%lld m=%d n=%d",        \
               (long long)batch, m, n);                                                                    \
    LQ_REQUIRE(c, batch == 0 || A != nullptr, LQ_ERR_ARG, "null input pointer")

// ---- kernel launches.  Every kernel of the linear-algebra entry points goes through launch<Kern> (launch_cluster<Kern>
// for one cluster of CTAs), which in this order
//   1. sets the kernel's attributes before its first launch on each device, if any are requested;
//   2. launches on stream st;
//   3. checks the launch with cudaGetLastError;
//   4. adds 1 to c->launches, the count lq_kernel_launches reports.
// opt_in_smem: 0 requests nothing, > 0 opts the kernel in to that many bytes of dynamic shared memory, SMEM_OPT_IN_REST
// to the device's opt-in maximum minus the kernel's static shared memory.  Cluster launches also allow cluster sizes
// beyond the portable 8.  The latch is keyed on the kernel itself, not on its type: kernels with the same signature
// (small_hh_kernel<0> and <1>) each need their own attribute.  Two host threads (two contexts) may race to the first
// launch: both then set the (idempotent) attribute and both publish the flag -- no torn state, no lock on the hot path.
// Devices beyond the table are configured on every launch.
struct DeviceLatch {
    std::atomic<unsigned char> f[64];
    bool test(int d) const { return d >= 0 && d < 64 && f[d].load(std::memory_order_acquire) != 0; }
    void set(int d) {
        if (d >= 0 && d < 64) f[d].store(1, std::memory_order_release);
    }
};

constexpr int SMEM_OPT_IN_REST = -1;

template <auto Kern>
int set_attributes_once(Ctx* c, int opt_in_smem, bool cluster) {
    if (opt_in_smem == 0 && !cluster) return LQ_OK;
    static DeviceLatch configured;
    if (configured.test(c->device)) return LQ_OK;
    if (opt_in_smem == SMEM_OPT_IN_REST) {
        cudaFuncAttributes fa{};
        LQ_CUDA(c, cudaFuncGetAttributes(&fa, Kern));
        opt_in_smem = c->max_smem - (int)fa.sharedSizeBytes;
    }
    if (opt_in_smem != 0)
        LQ_CUDA(c, cudaFuncSetAttribute(Kern, cudaFuncAttributeMaxDynamicSharedMemorySize, opt_in_smem));
    if (cluster) LQ_CUDA(c, cudaFuncSetAttribute(Kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    configured.set(c->device);
    return LQ_OK;
}

template <auto Kern, typename... Args>
int launch(Ctx* c, dim3 grid, dim3 block, size_t smem, cudaStream_t st, int opt_in_smem, Args... args) {
    LQ_TRY(set_attributes_once<Kern>(c, opt_in_smem, false));
    Kern<<<grid, block, smem, st>>>(args...);
    LQ_CHECK_LAUNCH(c);
    c->launches++;
    return LQ_OK;
}

// one cluster of cs CTAs (threads each, no dynamic shared memory) on the context stream
template <auto Kern, typename... Args>
int launch_cluster(Ctx* c, int cs, int threads, Args... args) {
    LQ_TRY(set_attributes_once<Kern>(c, 0, true));
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(cs);
    cfg.blockDim = dim3(threads);
    cfg.dynamicSmemBytes = 0;
    cfg.stream = c->stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = cs;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    LQ_CUDA(c, cudaLaunchKernelEx(&cfg, Kern, args...));
    c->launches++;
    return LQ_OK;
}

// ---- comm.cu
int comm_allreduce_sum(Ctx* c, double* buf, long long count);
int comm_allgather(Ctx* c, const double* send, double* recv, long long count_per_rank);

}  // namespace lq

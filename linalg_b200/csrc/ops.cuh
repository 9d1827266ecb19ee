// Internal (device-pointer) operations shared between the translation units.
#pragma once

#include "ctx.cuh"

namespace lq {

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

// ---- tallskinny.cu
int gram(Ctx* c, const double* A, long long m, int n, double* G);  // G = A^T A
// psd: the caller guarantees a positive semi-definite G (a Gram matrix): a well-conditioned one then gets its eigenvectors as
// the normalised converged columns b_i = lambda_i v_i instead of replaying the rotation log
int eigh_jacobi(Ctx* c, const double* G, int n, double* lambda_desc, double* V, bool psd = false);
int svd_gram_local(Ctx* c, const double* A, long long m, int n, double tol, double* U, double* s, double* Vt,
                   int* rank_host, bool sharded);
int tsqr_local(Ctx* c, const double* A, long long m, int n, double* Q, double* R, bool sharded);

// ---- batched (api_batched.cu).  qr32: 32 x 32 matrices go to the batched 32 x 32 kernel; false keeps them on the
// one-CTA kernel (the single-matrix entry point)
int hh_qr_batched_stream(Ctx* c, cudaStream_t st, const double* A, long long batch, int m, int n, double* Q,
                         double* R, bool qr32);

// Launch of a batched-family kernel on stream st.  attr_smem > 0 opts the kernel in to that many bytes of dynamic shared
// memory before its first launch on each device.  The latch is keyed on the kernel itself, not on its type: kernels with
// the same signature (small_hh_kernel<0> and <1>) each need their own attribute.
template <auto Kern, typename... Args>
int launch_batched(Ctx* c, cudaStream_t st, long long blocks, int threads, size_t smem, int attr_smem, Args... args) {
    if (attr_smem > 0) {
        static DeviceLatch configured;
        if (!configured.test(c->device)) {
            LQ_CUDA(c, cudaFuncSetAttribute(Kern, cudaFuncAttributeMaxDynamicSharedMemorySize, attr_smem));
            configured.set(c->device);
        }
    }
    Kern<<<(unsigned)blocks, threads, smem, st>>>(args...);
    LQ_CHECK_LAUNCH(c);
    LQ_COUNT_LAUNCH(c);
    return LQ_OK;
}

// ---- comm.cu
int comm_allreduce_sum(Ctx* c, double* buf, long long count);
int comm_allgather(Ctx* c, const double* send, double* recv, long long count_per_rank);

}  // namespace lq

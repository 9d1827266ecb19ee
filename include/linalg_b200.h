/* linalg_b200 -- C ABI of the B200-native dense-factorisation hot path.
 *
 * Drop-in boundary for BrantleighBunting/linalg's QR / least-squares / A^T A-SVD path.
 * The reference has no FFI of its own (pure Python + NumPy, SURVEY.md section 8b); each entry
 * point below replaces the Python function cited next to it, which the reference-side ctypes
 * stub in INTEGRATION.md binds 1:1.
 *
 * Conventions
 *   - all matrices are float64, row-major (C order), densely packed; batched arrays are
 *     (batch, rows, cols) with the batch index slowest -- exactly a C-contiguous NumPy array.
 *   - return value: 0 ok; < 0 argument / shape error (Python shim raises ValueError);
 *     > 0 CUDA (1000 + cudaError_t) or NCCL (5000 + ncclResult_t) failure (RuntimeError).
 *     lq_last_error() gives the text.  There is NO CPU fallback anywhere in this library.
 *   - "_dev" entry points take DEVICE pointers and enqueue on the context's stream without
 *     synchronising; the plain entry points take HOST pointers, copy in, run, copy out and
 *     return when the outputs are complete.
 *   - a context owns one device, one stream, its scratch memory and (optionally) one NCCL
 *     communicator; calls on one context must be serialised by the caller.
 *   - data-dependent failures (a linearly dependent column in MGS, linalg/qr.py:40-41) are
 *     reported per matrix in info[] (0 = fine, j+1 = first failing column); the shim raises
 *     the reference's ValueError.
 */
#ifndef LINALG_B200_H_
#define LINALG_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct lq_ctx lq_ctx;

/* ---- lifecycle ------------------------------------------------------------------------- */
const char* lq_version(void);
int lq_device_count(int* count);
int lq_create(int device, lq_ctx** out);
int lq_destroy(lq_ctx* ctx);
const char* lq_last_error(lq_ctx* ctx); /* ctx may be NULL: last error of a failed lq_create */
/* props[0]=SM count, [1]=cc major, [2]=cc minor, [3]=max dyn smem per block, [4]=SM clock kHz,
 * [5]=total global memory MiB, [6]=L2 bytes, [7]=max cluster size usable by the panel kernel */
int lq_device_props(lq_ctx* ctx, int64_t props[8]);

/* ---- memory / stream / timing ------------------------------------------------------------ */
int lq_malloc(lq_ctx* ctx, size_t bytes, void** dptr);
int lq_free(lq_ctx* ctx, void* dptr);
int lq_host_alloc(size_t bytes, void** hptr); /* pinned host memory */
int lq_host_free(void* hptr);
int lq_memcpy_h2d(lq_ctx* ctx, void* dst, const void* src, size_t bytes); /* async on ctx stream */
int lq_memcpy_d2h(lq_ctx* ctx, void* dst, const void* src, size_t bytes); /* async on ctx stream */
int lq_memcpy_d2d(lq_ctx* ctx, void* dst, const void* src, size_t bytes);
int lq_memset(lq_ctx* ctx, void* dst, int value, size_t bytes);
int lq_sync(lq_ctx* ctx);
int lq_event_record(lq_ctx* ctx, int slot);                       /* slot 0..15, on ctx stream */
int lq_event_elapsed_ms(lq_ctx* ctx, int slot_a, int slot_b, float* ms); /* syncs on slot_b */
int lq_flush_l2(lq_ctx* ctx);        /* overwrite a 256 MiB scratch buffer (> 126 MB L2) */
/* kernels the linear-algebra entry points launched on ctx so far, each counted once by the launch helper that launched it
 * (a CUDA-graph replay adds the kernels it holds); the measurement utilities lq_probe and lq_flush_l2 are not counted */
int64_t lq_kernel_launches(lq_ctx* ctx);

/* diagnostics: kernel-selection switches of one context.  name is the LINALG_B200_<NAME> environment variable without
 * its prefix ("TSQR_HOUSEHOLDER", "JACOBI_TWO_SIDED"); any other name returns LQ_ERR_ARG.  The environment only gives
 * the initial value at lq_create, hot entry points never call getenv. */
int lq_set_option(lq_ctx* ctx, const char* name, int value);

/* ---- a1: householder_qr  (linalg/qr.py:52-100) ------------------------------------------- */
/* A (batch, m, n) -> Q (batch, m, n), R (batch, n, n); requires m >= n >= 1.
 * variant: must be 0 (the library's kernel for each shape); any other value returns LQ_ERR_ARG.  The argument is kept
 * for ABI compatibility. */
int lq_householder_qr_batched_dev(lq_ctx* ctx, const double* A, int64_t batch, int m, int n, double* Q, double* R,
                                  int variant);
int lq_householder_qr_batched(lq_ctx* ctx, const double* A, int64_t batch, int m, int n, double* Q, double* R);
/* single (possibly large) matrix: blocked compact-WY Householder.
 * lq_householder_qr_dev replays its multi-stream launch schedule as a CUDA graph from the third call with the same shape AND the
 * same three device pointers (first call: plain launches, second: capture; up to 8 shapes are cached per context, one of them
 * larger than 2048^2).  The graph holds pointers, not data: the buffers' contents may change between calls.  Results are bit
 * for bit those of the plain launches; LINALG_B200_NO_GRAPH=1 disables the replay. */
int lq_householder_qr_dev(lq_ctx* ctx, const double* A, int m, int n, double* Q, double* R);
int lq_householder_qr(lq_ctx* ctx, const double* A, int m, int n, double* Q, double* R);

/* ---- a2: qr = modified Gram-Schmidt  (linalg/qr.py:14-49) --------------------------------- */
int lq_mgs_qr_batched_dev(lq_ctx* ctx, const double* A, int64_t batch, int m, int n, int reorth, double* Q,
                          double* R, int32_t* info);
int lq_mgs_qr_batched(lq_ctx* ctx, const double* A, int64_t batch, int m, int n, int reorth, double* Q, double* R,
                      int32_t* info);
int lq_mgs_qr_dev(lq_ctx* ctx, const double* A, int m, int n, int reorth, double* Q, double* R, int32_t* info);
int lq_mgs_qr(lq_ctx* ctx, const double* A, int m, int n, int reorth, double* Q, double* R, int32_t* info);

/* ---- a3: least_squares_householder_qr  (linalg/qr.py:122-134) ------------------------------ */
/* A (batch, m, n), B (batch, m, nrhs) -> X (batch, n, nrhs) */
int lq_lstsq_householder_batched_dev(lq_ctx* ctx, const double* A, const double* B, int64_t batch, int m, int n,
                                     int nrhs, double* X);
int lq_lstsq_householder_batched(lq_ctx* ctx, const double* A, const double* B, int64_t batch, int m, int n,
                                 int nrhs, double* X);
/* the same with a per-system singularity report: info[b] = 0, or 1 + the first column whose R[j][j] is exactly 0 -- the
 * case in which the reference's np.linalg.solve raises LinAlgError("Singular matrix") (linalg/qr.py:134); the shim raises the
 * same.  Every route (warp-per-system, streaming, one-CTA and blocked) fills it; info may be NULL. */
int lq_lstsq_householder_batched_info_dev(lq_ctx* ctx, const double* A, const double* B, int64_t batch, int m, int n,
                                          int nrhs, double* X, int32_t* info);
int lq_lstsq_householder_batched_info(lq_ctx* ctx, const double* A, const double* B, int64_t batch, int m, int n,
                                      int nrhs, double* X, int32_t* info);

/* ---- a4: least_squares_qr (MGS)  (linalg/qr.py:103-119) ------------------------------------ */
int lq_lstsq_mgs_batched_dev(lq_ctx* ctx, const double* A, const double* B, int64_t batch, int m, int n, int nrhs,
                             double* X, int32_t* info);
int lq_lstsq_mgs_batched(lq_ctx* ctx, const double* A, const double* B, int64_t batch, int m, int n, int nrhs,
                         double* X, int32_t* info);

/* ---- a5: svd via the A^T A eigen-route  (linalg/svd.py:10-82), m >= n ------------------------- */
/* U (m, n), s (n) descending, Vt (n, n); *rank = #(s > tol).  Columns of U beyond rank are
 * left ZERO here; the shim completes them (svd.py:67-76) with lq_svd_complete.
 * Non-finite input: a NaN or Inf in A, or a finite A whose A^T A overflows, gives s = NaN throughout, Vt = I and rank 0
 * (lq_eigh_dev's contract; sigma of a NaN eigenvalue is NaN, never 0), with no error: the reference raises for some such
 * shapes and returns NaN singular values for the others, never an all-finite s.  This holds for lq_svd_gram_batched too. */
int lq_svd_gram_dev(lq_ctx* ctx, const double* A, int64_t m, int n, double tol, double* U, double* s, double* Vt,
                    int* rank_host);
int lq_svd_gram(lq_ctx* ctx, const double* A, int64_t m, int n, double tol, double* U, double* s, double* Vt,
                int* rank_host);
/* the same for every matrix of a batch: A (batch, m, n) -> U (batch, m, n), s (batch, n), Vt (batch, n, n), rank (batch)
 * for m >= n >= 1; U columns beyond rank are left ZERO (completed by the shim, as for lq_svd_gram).  n <= 32 and
 * m <= 4096: one warp per matrix (two-sided Jacobi on the scaled Gram matrix, the rotation test of the single path);
 * other shapes: lq_svd_gram matrix by matrix, bit for bit.  The route depends on (m, n) only. */
int lq_svd_gram_batched_dev(lq_ctx* ctx, const double* A, int64_t batch, int m, int n, double tol, double* U, double* s,
                            double* Vt, int32_t* rank);            /* device pointers */
int lq_svd_gram_batched(lq_ctx* ctx, const double* A, int64_t batch, int m, int n, double tol, double* U, double* s,
                        double* Vt, int32_t* rank);                /* host pointers: the two-lane chunked pipeline */
/* svd.py:67-76: complete U (HOST, m x n, first `rank` columns valid) with an orthonormal basis of the
 * complement built from the caller-drawn candidates Z (HOST, m x (n - rank)); all arithmetic on device. */
int lq_svd_complete(lq_ctx* ctx, double* U, int64_t m, int n, int rank, const double* Z);
/* the same with the candidates generated ON THE DEVICE from `seed` (Philox4x32-10 + Box-Muller; deterministic, no m x (n-rank)
 * upload).  The reference draws them from the global np.random (svd.py:69), i.e. it is not reproducible there; only the
 * invariants of the completion are pinned by its tests (tests/test_svd.py:60-79). */
int lq_svd_complete_seeded(lq_ctx* ctx, double* U, int64_t m, int n, int rank, uint64_t seed);
/* `count` standard-normal doubles of that generator into device memory (a function of (seed, index) only) */
int lq_random_normal_dev(lq_ctx* ctx, double* out, int64_t count, uint64_t seed);
/* building blocks (device pointers) */
int lq_gram_dev(lq_ctx* ctx, const double* A, int64_t m, int n, double* G);          /* G = A^T A (n x n) */
/* Eigen-decomposition of a symmetric POSITIVE SEMI-DEFINITE matrix (the Gram / covariance matrices of svd.py:42,46 and
 * pca): eigenvalues descending, eigenvectors in the columns of V.  n <= 128: one-sided Jacobi on the columns of G (it
 * orthogonalises them, i.e. diagonalises G^2: eigenvalues of equal magnitude and opposite sign would not be separated,
 * which cannot happen for PSD input); 128 < n <= 2048: two-sided Jacobi (any symmetric matrix).  Input range: any finite
 * G whose largest |diagonal| entry is normal (2^-1022 to 2^1024); both kernels work on G scaled by a power of two to a
 * largest diagonal entry in [1, 2), so the result scales with G, bit for bit, as long as no entry of the scaled G is
 * subnormal.  A G with a NaN or infinite entry returns NaN for every eigenvalue and V = I, and is not an error (the
 * reference's eigh raises for some such n and returns n - 1 or n NaN values for the others); lambda_desc is sorted with NaN
 * first, as np.argsort(lam)[::-1] puts it, and every element of lambda_desc and V is written for any input
 * (tests/test_gpu_nonfinite.py). */
int lq_eigh_dev(lq_ctx* ctx, const double* G, int n, double* lambda_desc, double* V);
/* row-major C = a op(A) op(B) + b C.  With b = 0, C is not read: it may hold anything, NaN and Inf included. */
int lq_gemm_dev(lq_ctx* ctx, int transa, int transb, int64_t m, int n, int k, double alpha, const double* A,
                int lda, const double* B, int ldb, double beta, double* C, int ldc);

/* ---- a7: TSQR for tall-skinny matrices, diag(R) > 0 (the MGS convention) ------------------------ */
int lq_tsqr_dev(lq_ctx* ctx, const double* A, int64_t m, int n, double* Q, double* R);
int lq_tsqr(lq_ctx* ctx, const double* A, int64_t m, int n, double* Q, double* R);
/* least squares on the same pipeline: X (n, nrhs) = argmin ||A X - B||_F for A (m, n), B (m, nrhs); m < 2^31 per device.
 * info: 0, or 1 + the first column whose R[j][j] is exactly 0 (the contract of lq_lstsq_householder_batched_info).
 * Routes: n <= 128 and m >= 4n: CholeskyQR2 that never forms Q (G1 = A^T A -> R1, Q1 = A R1^-1, [G2 | C] = Q1^T [Q1 | B] in one
 * pass for even n, nrhs <= 32, m >= 1024 -> R2, X = (R2 R1)^-1 R2^-T C), accepted under TSQR's cond(A)^2 < 1e10 verdict.
 * Otherwise (ill-conditioned, m < 4n, n > 128 or TSQR_HOUSEHOLDER set) the lq_lstsq_householder_batched_info route. */
int lq_lstsq_tsqr_dev(lq_ctx* ctx, const double* A, int64_t m, int n, const double* B, int nrhs, double* X, int32_t* info);
int lq_lstsq_tsqr(lq_ctx* ctx, const double* A, int64_t m, int n, const double* B, int nrhs, double* X, int32_t* info);

/* ---- multi-GPU: one process (context) per GPU, NCCL over NVLink ---------------------------------- */
int lq_comm_unique_id(void* id128);                                     /* 128 bytes, from rank 0 */
int lq_comm_init(lq_ctx* ctx, int nranks, int rank, const void* id128); /* collective */
int lq_comm_destroy(lq_ctx* ctx);
int lq_comm_allreduce_sum(lq_ctx* ctx, double* dbuf, int64_t count);    /* in place, ctx stream */
int lq_comm_allgather(lq_ctx* ctx, const double* dsend, double* drecv, int64_t count_per_rank);
/* row-sharded: every rank passes its (m_local, n) block; R / s / Vt are replicated */
int lq_tsqr_sharded_dev(lq_ctx* ctx, const double* A_local, int64_t m_local, int n, double* Q_local, double* R);
int lq_svd_gram_sharded_dev(lq_ctx* ctx, const double* A_local, int64_t m_local, int n, double tol, double* U_local,
                            double* s, double* Vt, int* rank_host);
/* row-sharded least squares, n <= 128: every rank passes its (m_local, n) block of A and (m_local, nrhs) block of B; X (n, nrhs)
 * and info come back replicated, bitwise identical on every rank.  CholeskyQR2 as in lq_lstsq_tsqr_dev (one all-reduce per
 * pass); when its verdict fails or TSQR_HOUSEHOLDER is set, the Householder reduction tree of [A_local | B_local] with an
 * all-gather of the local R factors, whose top n rows are [R | Q^T B] (needs n + nrhs <= 128 and m_local >= n + nrhs on every
 * rank; otherwise every rank returns the same error). */
int lq_lstsq_tsqr_sharded_dev(lq_ctx* ctx, const double* A_local, int64_t m_local, int n, const double* B_local, int nrhs,
                              double* X, int32_t* info);

/* ---- roofline probes (bench.py) --------------------------------------------------------------------- */
/* kind 0: FP64 FMA (DFMA) peak, 1: FP64 tensor (DMMA m16n8k8) peak, 3: both pipes mixed [TFLOP/s];
 * 2: device copy [GB/s]; 4: dependent DFMA latency [cycles]; 10..16: accuracy of the MUFU seeds and
 * Newton-refined rcp / rsqrt / sqrt used by the kernels [max relative error]. */
int lq_probe(lq_ctx* ctx, int kind, double* result);
/* diagnostics: one 32-column panel factorisation of the blocked path with an explicit kernel version
 * (0 default, 1 barrier.cluster kernel, 3 st.async kernel with 256 rows per CTA); any other version returns LQ_ERR_ARG */
int lq_debug_panel(lq_ctx* ctx, double* A, int lda, double* V, int ldv, double* T, int ldt, int mp, int nb, int version);
/* the same with clock64() stamps of the column-step phases: trace[2 warps][32 columns][8 phases] (device pointer) */
int lq_debug_panel_trace(lq_ctx* ctx, double* A, int lda, double* V, int ldv, double* T, int ldt, int mp, long long* trace);

#ifdef __cplusplus
}
#endif
#endif /* LINALG_B200_H_ */

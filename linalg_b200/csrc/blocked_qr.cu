// K4: blocked compact-WY Householder QR of one (possibly large) matrix -- linalg/qr.py:52-100.
//
// Two-level right-looking factorisation.  Outer block NB = 128 columns; inside it, 32-column
// panels are factored by the register/DSMEM cluster kernel (panel.cuh), the rest of the outer
// block is updated with the panel's own T, then the 128-wide block reflector I - V T V^T
// (T from the Gram matrix V^T V) updates the trailing matrix with three FP64 tensor-core GEMMs:
//     W  = V^T C          (TN, K = rows)
//     W2 = T^T W          (TN, K = 128)
//     C -= V W2           (NN, K = 128)
// Q is formed by applying the block reflectors to the identity in reverse order.  The working
// copies are padded to a multiple of 32 columns (zero columns are "skipped" reflectors, exactly
// the reference's  ||x|| < 1e-12  branch), so every GEMM operand is 16-byte aligned.
#include <algorithm>
#include <vector>

#include "../../include/linalg_b200.h"
#include "ops.cuh"
#include "panel.cuh"
#include "panel2.cuh"

namespace lq {

namespace {

constexpr int NB_OUT = 128;
constexpr int NB_IN = 32;

// ------------------------------------------------------------------ small helper kernels
__global__ void __launch_bounds__(256) pad_copy_kernel(const double* __restrict__ src, int lds, double* __restrict__ dst,
                                                       int ldd, long long rows, int cols_src, int cols_dst) {
    const long long total = rows * cols_dst;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const long long i = e / cols_dst;
        const int j = (int)(e - i * cols_dst);
        dst[i * ldd + j] = (j < cols_src) ? src[i * lds + j] : 0.0;
    }
}
__global__ void __launch_bounds__(256) unpad_copy_kernel(const double* __restrict__ src, int lds, double* __restrict__ dst,
                                                         int ldd, long long rows, int cols) {
    const long long total = rows * cols;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const long long i = e / cols;
        const int j = (int)(e - i * cols);
        dst[i * ldd + j] = src[i * lds + j];
    }
}
__global__ void __launch_bounds__(256) extract_upper_kernel(const double* __restrict__ src, int lds, double* __restrict__ R,
                                                            int n) {
    const long long total = (long long)n * n;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const int i = (int)(e / n), j = (int)(e - (long long)i * n);
        R[e] = (j >= i) ? src[(long long)i * lds + j] : 0.0;  // strict lower triangle exact zeros (qr.py:97)
    }
}
__global__ void __launch_bounds__(256) set_identity_kernel(double* __restrict__ Q, int ldq, long long rows, int cols) {
    const long long total = rows * cols;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const long long i = e / cols;
        const int j = (int)(e - i * cols);
        Q[i * ldq + j] = (i == j) ? 1.0 : 0.0;
    }
}

// Merge the 32 x 32 panel factors on the diagonal of T (kb x kb, kb = 32 * nblk <= 128) into the factor of
// the whole outer block, using the Gram matrix G = V^T V:  for column block b = 1 .. nblk-1
//     T[0:R, b] = -T[0:R, 0:R] * G[0:R, b] * T[b, b],   R = 32 b
// (the block form of LAPACK dlarft; V1 := the first R reflectors).  One CTA, everything in shared memory.
template <int KBC>  // KBC = 128: compile-time block size (shifts instead of integer divisions); 0: runtime kb
__global__ void __launch_bounds__(1024) merge_t_kernel(const double* __restrict__ G, int ldg, double* __restrict__ T, int ldt,
                                                       int kb_rt) {
    const int kb = KBC ? KBC : kb_rt;
    extern __shared__ double sh[];
    double* Ts = sh;               // [128][129]
    double* Xs = Ts + 128 * 129;   // [96][33]
    double* Ys = Xs + 96 * 33;     // [96][33]
    const int tid = threadIdx.x, nt = blockDim.x;
    const int nblk = kb / 32;
    // only the diagonal 32 x 32 blocks are read: 4 independent loads per thread
    for (int e = tid; e < kb * kb; e += nt) Ts[(e / kb) * 129 + (e % kb)] = 0.0;
    __syncthreads();
    for (int e = tid; e < nblk * 32 * 32; e += nt) {
        const int b = e >> 10, i = (e >> 5) & 31, k = e & 31;
        if (k >= i) Ts[(32 * b + i) * 129 + 32 * b + k] = T[(long long)(32 * b + i) * ldt + 32 * b + k];
    }
    __syncthreads();
    for (int b = 1; b < nblk; ++b) {
        const int R = 32 * b, c0 = 32 * b;
        for (int e = tid; e < R * 32; e += nt) {
            const int i = e >> 5, cc = e & 31;
            Xs[i * 33 + cc] = G[(long long)i * ldg + c0 + cc];
        }
        __syncthreads();
        for (int e = tid; e < R * 32; e += nt) {
            const int i = e >> 5, cc = e & 31;
            double a0 = 0.0, a1 = 0.0;
            int k = i;
            for (; k + 2 <= R; k += 2) {
                a0 = fma(Ts[i * 129 + k], Xs[k * 33 + cc], a0);
                a1 = fma(Ts[i * 129 + k + 1], Xs[(k + 1) * 33 + cc], a1);
            }
            if (k < R) a0 = fma(Ts[i * 129 + k], Xs[k * 33 + cc], a0);
            Ys[i * 33 + cc] = a0 + a1;
        }
        __syncthreads();
        for (int e = tid; e < R * 32; e += nt) {
            const int i = e >> 5, cc = e & 31;
            double acc = 0.0;
            for (int k = 0; k <= cc; ++k) acc = fma(Ys[i * 33 + k], Ts[(c0 + k) * 129 + c0 + cc], acc);
            Ts[i * 129 + c0 + cc] = -acc;
        }
        __syncthreads();
    }
    for (int e = tid; e < kb * kb; e += nt) {
        const int i = e / kb, k = e - i * kb;
        T[(long long)i * ldt + k] = Ts[i * 129 + k];
    }
}
constexpr size_t MERGE_T_SMEM = (128 * 129 + 2 * 96 * 33) * sizeof(double);

// ------------------------------------------------------------------ generic (any height) panel, BLAS-2, multi-launch
// Used only when the panel does not fit the cluster kernel (mp > 16 * 512 rows).  Column j:
//   k1: per-CTA partial  x^T P[:, c]  for all c -> atomicAdd into acc[0:nb]; pivot row copied to acc[nb:2nb]
//   k2: every CTA forms alpha, v0, beta and updates its rows; CTA 0 also maintains T_u, beta, v0, rdiag
struct GPanelState {
    double acc[64];     // [0:32) dots, [32:64) pivot row
    double Tt[32 * 32]; // Tt[k*32+i] = T_u[i][k]
    double beta[32], v0[32], rdiag[32];
};
__global__ void __launch_bounds__(256) gpanel_dots_kernel(const double* __restrict__ A, int lda, int mp, int nb, int j,
                                                          GPanelState* st, int rows_per_cta) {
    __shared__ double red[8][32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int r0 = blockIdx.x * rows_per_cta;
    const int r1 = min(mp, r0 + rows_per_cta);
    double d = 0.0;
    for (int r = max(r0, j) + w; r < r1; r += 8) {
        const double x = A[(long long)r * lda + j];
        if (lane < nb) d = fma(x, A[(long long)r * lda + lane], d);
    }
    red[w][lane] = d;
    __syncthreads();
    if (w == 0) {
        double s = 0.0;
        for (int ww = 0; ww < 8; ++ww) s += red[ww][lane];
        if (lane < nb && s != 0.0) atomicAdd(&st->acc[lane], s);
        if (j >= r0 && j < r1 && lane < nb) st->acc[32 + lane] = A[(long long)j * lda + lane];
    }
}
__global__ void __launch_bounds__(256) gpanel_update_kernel(double* __restrict__ A, int lda, int mp, int nb, int j,
                                                            GPanelState* st, int rows_per_cta) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int r0 = blockIdx.x * rows_per_cta;
    const int r1 = min(mp, r0 + rows_per_cta);
    const double tot = (lane < nb) ? st->acc[lane] : 0.0;
    const double prow = (lane < nb && j < mp) ? st->acc[32 + lane] : 0.0;
    const double ss = __shfl_sync(0xffffffffu, tot, j);
    const double x0 = __shfl_sync(0xffffffffu, prow, j);
    const double nrm = sqrt(fmax(ss, 0.0));
    const bool skip = nrm < kEps;
    const double alpha = copysign(nrm, x0);
    const double v0 = x0 + alpha;
    const double beta = skip ? 0.0 : 1.0 / (nrm * fabs(v0));
    const double gl = fma(alpha, prow, tot);
    const double sc = (lane > j && lane < nb) ? beta * gl : 0.0;
    for (int r = max(r0, j) + w; r < r1; r += 8) {
        double x = A[(long long)r * lda + j];
        if (r == j) x = v0;
        if (lane > j && lane < nb) A[(long long)r * lda + lane] = fma(-sc, x, A[(long long)r * lda + lane]);
    }
    if (blockIdx.x == 0 && w == 0) {
        // T column (same recurrence as the cluster kernel) -- uses the totals before they are cleared
        double acc = 0.0;
        __shared__ double gb[32];
        gb[lane] = gl;
        __syncwarp();
        for (int k = 0; k < j; ++k) acc = fma(st->Tt[k * 32 + lane], gb[k], acc);
        if (lane < j) st->Tt[j * 32 + lane] = -beta * acc;
        if (lane == j) st->Tt[j * 32 + lane] = beta;
        if (lane == 0) {
            st->beta[j] = beta;
            st->v0[j] = v0;
            st->rdiag[j] = skip ? x0 : -alpha;
        }
    }
}
__global__ void __launch_bounds__(64) gpanel_clear_kernel(GPanelState* st, int all) {
    const int t = threadIdx.x;
    st->acc[t] = 0.0;
    if (all) {
        for (int e = t; e < 32 * 32; e += 64) st->Tt[e] = 0.0;
        if (t < 32) st->beta[t] = 0.0, st->v0[t] = 0.0, st->rdiag[t] = 0.0;
    }
}
__global__ void __launch_bounds__(256) gpanel_store_kernel(double* __restrict__ A, int lda, double* __restrict__ V, int ldv,
                                                           double* __restrict__ T, int ldt, int mp, int nb,
                                                           const GPanelState* st) {
    const long long total = (long long)mp * nb;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const int row = (int)(e / nb), c = (int)(e - (long long)row * nb);
        const double bt = st->beta[c];
        const double rn = sqrt(0.5 * bt);
        double vv;
        if (row > c) vv = A[(long long)row * lda + c] * rn;
        else if (row == c) vv = st->v0[c] * rn;
        else vv = 0.0;
        V[(long long)row * ldv + c] = vv;
        if (row == c) A[(long long)row * lda + c] = st->rdiag[c];
    }
    if (blockIdx.x == 0) {
        for (int e = threadIdx.x; e < nb * nb; e += blockDim.x) {
            const int i = e / nb, k = e - i * nb;
            const double bi = st->beta[i], bk = st->beta[k];
            double val = 0.0;
            if (i <= k && bi > 0.0 && bk > 0.0) val = st->Tt[k * 32 + i] * 2.0 / sqrt(bi * bk);
            T[(long long)i * ldt + k] = val;
        }
    }
}

int panel_generic(Ctx* c, double* A, int lda, double* V, int ldv, double* T, int ldt, int mp, int nb) {
    DevBuf stb;
    LQ_TRY(stb.alloc(c, sizeof(GPanelState)));
    GPanelState* st = stb.as<GPanelState>();
    const int ctas = std::max(1, std::min(c->sm_count * 2, (mp + 255) / 256));
    const int rpc = (mp + ctas - 1) / ctas;
    LQ_TRY(launch<gpanel_clear_kernel>(c, 1, 64, 0, c->stream, 0, st, 1));
    for (int j = 0; j < nb; ++j) {
        LQ_TRY(launch<gpanel_dots_kernel>(c, ctas, 256, 0, c->stream, 0, A, lda, mp, nb, j, st, rpc));
        LQ_TRY(launch<gpanel_update_kernel>(c, ctas, 256, 0, c->stream, 0, A, lda, mp, nb, j, st, rpc));
        LQ_TRY(launch<gpanel_clear_kernel>(c, 1, 64, 0, c->stream, 0, st, 0));
    }
    return launch<gpanel_store_kernel>(c, std::min(ctas, 64), 256, 0, c->stream, 0, A, lda, V, ldv, T, ldt, mp, nb, st);
}

// version: 0 = default choice (panels of up to 256 rows: the one-CTA SOLO kernel), 1 = barrier.cluster kernel (panel.cuh),
// 3 = st.async kernel (panel2.cuh) with 8 rows per lane (256 rows per CTA) wherever a cluster of it holds the panel
int panel_factor_v(Ctx* c, double* A, int lda, double* V, int ldv, double* T, int ldt, int mp, int nb, int version) {
    using Cfg = PanelCfg<4, 16>;
    const int maxcs = c->max_cluster;
    if (nb == P2_NB && version != 1) {
        // default: the 256-rows-per-CTA kernel whenever the panel fits a cluster of it (half the FP64 work per SM and
        // column); taller panels run next to the side stream's big GEMMs, where the barrier.cluster kernel measured
        // better in situ (tools/blocked_trace.py) than a 512-row st.async kernel, although that one won stand-alone
        if (version == 0 && mp <= Panel2Cfg<8>::ROWS_PER_CTA) {
            // one CTA, no cluster exchange: ~17 us instead of 48 us per panel of up to 256 rows
            return launch<panel2_cluster_kernel<8, false, true>>(c, 1, P2_THREADS, 0, c->stream, 0, A, lda, V, ldv, T, ldt, mp,
                                                                 (long long*)nullptr);
        }
        if (mp <= maxcs * Panel2Cfg<8>::ROWS_PER_CTA) {
            int cs = 1;
            while (cs * Panel2Cfg<8>::ROWS_PER_CTA < mp) cs *= 2;
            return launch_cluster<panel2_cluster_kernel<8, false>>(c, cs, P2_THREADS, A, lda, V, ldv, T, ldt, mp, (long long*)nullptr);
        }
    }
    int cs = 1;
    while (cs * Cfg::ROWS_PER_CTA < mp && cs < maxcs) cs *= 2;
    if (cs * Cfg::ROWS_PER_CTA < mp || nb > Cfg::NBMAX) return panel_generic(c, A, lda, V, ldv, T, ldt, mp, nb);
    return launch_cluster<panel_cluster_kernel<4, 16>>(c, cs, PANEL_THREADS, A, lda, V, ldv, T, ldt, mp, nb);
}

int panel_factor(Ctx* c, double* A, int lda, double* V, int ldv, double* T, int ldt, int mp, int nb) {
    return panel_factor_v(c, A, lda, V, ldv, T, ldt, mp, nb, 0);
}

// apply the block reflector  C <- (I - V op(T) V^T) C   to C (mk x nc, ldc); V (mk x kb, ldv); T (kb x kb, ldt)
// trans_t = true -> T^T (factorisation order H_kb ... H_1), false -> T (Q formation order H_1 ... H_kb)
int apply_block_reflector(Ctx* c, const double* V, int ldv, const double* T, int ldt, bool trans_t, int mk, int kb,
                          double* Cm, int ldc, int nc, double* W2) {
    if (nc <= 0 || kb <= 0 || mk <= 0) return LQ_OK;
    LQ_TRY(gemm_vtc_apply_t(c, kb, nc, mk, V, ldv, Cm, ldc, T, ldt, trans_t, W2));         // W2 = op(T) (V^T C)
    LQ_TRY(gemm(c, false, false, mk, nc, kb, -1.0, V, ldv, W2, nc, 1.0, Cm, ldc));         // C -= V W2
    return LQ_OK;
}

struct Factored {
    DevBuf Tall;     // per outer block: NB_OUT x NB_OUT
    int nblocks = 0;
};

// run a scope of library calls on another stream of the context (the host side is single threaded per context)
struct StreamScope {
    Ctx* c;
    cudaStream_t saved;
    StreamScope(Ctx* ctx, cudaStream_t s) : c(ctx), saved(ctx->stream) { c->stream = s; }
    ~StreamScope() { c->stream = saved; }
};
struct EventPool {
    std::vector<cudaEvent_t> ev;
    ~EventPool() {
        for (cudaEvent_t e : ev) cudaEventDestroy(e);
    }
    bool timing = false;
    int make(Ctx* c, cudaEvent_t* out) {
        LQ_CUDA(c, cudaEventCreateWithFlags(out, timing ? cudaEventDefault : cudaEventDisableTiming));
        ev.push_back(*out);
        return LQ_OK;
    }
};

// A (m x npad, lda) in place; V (m x npad, ldv) zero-initialised by the caller; npad % 32 == 0.
//
// Look-ahead schedule over two streams.  The panel chain of outer block b (four cluster-panel kernels, the
// narrow updates between them, Gram + T merge) is latency bound and uses 16 SMs; the trailing update with
// block b is throughput bound.  So after block b is factored, the context stream (high priority) applies it
// to the columns of block b+1 only and goes straight on to factor block b+1, while the side stream applies
// block b to all the remaining columns (and to the right-hand sides).  Dependencies:
//     side:  rest(b)  after panel(b)                    [event ev_panel[b]]   and after rest(b-1) [stream order]
//     main:  next(b)  after rest(b-1)                   [event ev_rest[b-1]]  (block b+1's columns were in rest(b-1))
int factor_padded(Ctx* c, double* A, int lda, int m, int npad, int nfac, double* V, int ldv, double* B, int ldb,
                  int nrhs_pad, Factored* keep) {
    const int nblocks = (nfac + NB_OUT - 1) / NB_OUT;
    cudaStream_t s_main = c->stream, s_side = c->lane[0], s_aux = c->lane[1], s_merge = c->lane[2], s_side2 = c->lane[3];
    const bool lookahead = nblocks > 1;
    // Gram scratch of the T merge: one buffer per stream that may run a merge (main: blocks without panel-wise look-ahead,
    // e.g. the last one; merge stream: all the others) -- the two streams are not ordered against each other
    DevBuf Tloc, G, Gmerge, W2, W2s, W2s2;
    LQ_TRY(G.alloc(c, sizeof(double) * NB_OUT * NB_OUT));
    LQ_TRY(Gmerge.alloc(c, sizeof(double) * NB_OUT * NB_OUT));
    const int wcols = std::max(npad, nrhs_pad);
    LQ_TRY(W2.alloc(c, sizeof(double) * NB_OUT * (size_t)wcols));
    DevBuf W2a;  // scratch of the aux stream (panel-wise application to the next outer block)
    if (lookahead) {
        LQ_TRY(W2s.alloc(c, sizeof(double) * NB_OUT * (size_t)wcols));
        LQ_TRY(W2s2.alloc(c, sizeof(double) * NB_OUT * (size_t)wcols));
        LQ_TRY(W2a.alloc(c, sizeof(double) * NB_IN * (size_t)NB_OUT));
    }
    double* Tall;
    if (keep) {
        LQ_TRY(keep->Tall.alloc(c, sizeof(double) * NB_OUT * NB_OUT * (size_t)nblocks));
        keep->nblocks = nblocks;
        Tall = keep->Tall.as<double>();
    } else {
        LQ_TRY(Tloc.alloc(c, sizeof(double) * NB_OUT * NB_OUT * (size_t)nblocks));
        Tall = Tloc.as<double>();
    }
    LQ_CUDA(c, cudaMemsetAsync(Tall, 0, sizeof(double) * NB_OUT * NB_OUT * (size_t)nblocks, s_main));
    EventPool pool;
    // diagnostics (LINALG_B200_TRACE_BLOCKS=1): per outer block, when the panel chain, the next-block update and the
    // side stream's trailing update finished (ms since the start of the factorisation), printed to stderr
    const bool trace_blocks = lookahead && LQ_ENV_ONCE("LINALG_B200_TRACE_BLOCKS");
    pool.timing = trace_blocks;
    struct BlockTrace { cudaEvent_t panels = nullptr, chain = nullptr, next = nullptr, rest = nullptr; };
    std::vector<BlockTrace> btrace(trace_blocks ? nblocks : 0);
    cudaEvent_t ev_t0 = nullptr;
    cudaEvent_t ev_rest_prev = nullptr;   // completion of the trailing update that held the NEXT block's columns
    cudaEvent_t ev_rest_last[2] = {nullptr, nullptr};  // last trailing updates of the two column ranges (final join)
    // the trailing update runs on two independent column ranges (block reflectors act on columns independently), split
    // where the flops balance (3 s^2 - s^3 = 1): launch gaps, reductions and partial waves of one range are filled by the other
    const int rsplit = (lookahead && npad >= 6144) ? (int)(0.65 * npad) / NB_OUT * NB_OUT : 0;
    if (trace_blocks) {
        LQ_TRY(pool.make(c, &ev_t0));
        LQ_CUDA(c, cudaEventRecord(ev_t0, s_main));
    }
    if (lookahead) {
        // the scratch buffers of the side stream come from the main stream's pool allocation
        cudaEvent_t e0;
        LQ_TRY(pool.make(c, &e0));
        LQ_CUDA(c, cudaEventRecord(e0, s_main));
        LQ_CUDA(c, cudaStreamWaitEvent(s_side, e0, 0));
        LQ_CUDA(c, cudaStreamWaitEvent(s_aux, e0, 0));
        LQ_CUDA(c, cudaStreamWaitEvent(s_merge, e0, 0));
        LQ_CUDA(c, cudaStreamWaitEvent(s_side2, e0, 0));
    }
    for (int blk = 0; blk < nblocks; ++blk) {
        const int k0 = blk * NB_OUT;
        const int kb = std::min(NB_OUT, npad - k0);  // multiple of 32
        const int mk = m - k0;
        double* Tblk = Tall + (size_t)blk * NB_OUT * NB_OUT;
        if (mk <= 0) continue;
        const int nin = kb / NB_IN;
        const int ntr = npad - (k0 + kb);
        const int nnext = std::min(NB_OUT, ntr);
        const int nrest = ntr - nnext;
        double* Ctr = A + (size_t)k0 * lda + k0 + kb;
        // panel-wise look-ahead: every panel's own reflector (V_p, T_p) is applied to the columns of the NEXT outer
        // block on the aux stream as soon as the panel exists, in the shadow of the following panels, so the chain
        // never waits for the Gram matrix / T merge of the whole block (they move to the side stream, where only the
        // big trailing update and the Q formation need the merged T)
        const bool pw = lookahead && nnext > 0 && nin > 1;
        cudaEvent_t ev_aux_done = nullptr;
        for (int ip = 0; ip < nin; ++ip) {
            const int c0 = k0 + ip * NB_IN;
            const int mp = m - c0;
            if (mp <= 0) break;
            double* Ap = A + (size_t)c0 * lda + c0;
            double* Vp = V + (size_t)c0 * ldv + c0;
            double* Tp = Tblk + (size_t)ip * NB_IN * NB_OUT + ip * NB_IN;  // diagonal block of the outer T
            const int ldtp = NB_OUT;
            LQ_TRY(panel_factor(c, Ap, lda, Vp, ldv, Tp, ldtp, mp, NB_IN));
            if (pw) {
                cudaEvent_t ev_p;
                LQ_TRY(pool.make(c, &ev_p));
                LQ_CUDA(c, cudaEventRecord(ev_p, s_main));
                StreamScope aux(c, s_aux);
                LQ_CUDA(c, cudaStreamWaitEvent(s_aux, ev_p, 0));
                if (ip == 0 && ev_rest_prev) LQ_CUDA(c, cudaStreamWaitEvent(s_aux, ev_rest_prev, 0));  // block b+1's columns were in rest(b-1)
                LQ_TRY(apply_block_reflector(c, Vp, ldv, Tp, ldtp, true, mp, NB_IN, A + (size_t)c0 * lda + k0 + kb, lda, nnext,
                                             W2a.as<double>()));
                if (ip == nin - 1) {
                    LQ_TRY(pool.make(c, &ev_aux_done));
                    LQ_CUDA(c, cudaEventRecord(ev_aux_done, s_aux));
                }
            }
            const int nrem = k0 + kb - (c0 + NB_IN);
            if (nrem > 0)
                LQ_TRY(apply_block_reflector(c, Vp, ldv, Tp, ldtp, true, mp, NB_IN, Ap + NB_IN, lda, nrem,
                                             W2.as<double>()));
        }
        if (trace_blocks) {
            LQ_TRY(pool.make(c, &btrace[blk].panels));
            LQ_CUDA(c, cudaEventRecord(btrace[blk].panels, s_main));
        }
        const double* Vb = V + (size_t)k0 * ldv + k0;
        // the T factor of the whole outer block: on the stream that needs it first
        auto merge_block_t = [&](double* Gs) -> int {
            if (nin <= 1) return LQ_OK;
            LQ_TRY(gemm(c, true, false, kb, kb, mk, 1.0, Vb, ldv, Vb, ldv, 0.0, Gs, NB_OUT));  // G = V^T V
            if (kb == 128)
                return launch<merge_t_kernel<128>>(c, 1, 1024, MERGE_T_SMEM, c->stream, (int)MERGE_T_SMEM, Gs, NB_OUT, Tblk, NB_OUT, kb);
            return launch<merge_t_kernel<0>>(c, 1, 1024, MERGE_T_SMEM, c->stream, (int)MERGE_T_SMEM, Gs, NB_OUT, Tblk, NB_OUT, kb);
        };
        if (!lookahead) {
            LQ_TRY(merge_block_t(G.as<double>()));
            if (ntr > 0)
                LQ_TRY(apply_block_reflector(c, Vb, ldv, Tblk, NB_OUT, true, mk, kb, Ctr, lda, ntr, W2.as<double>()));
            if (B && nrhs_pad > 0)
                LQ_TRY(apply_block_reflector(c, Vb, ldv, Tblk, NB_OUT, true, mk, kb, B + (size_t)k0 * ldb, ldb, nrhs_pad,
                                             W2.as<double>()));
            continue;
        }
        cudaEvent_t ev_panel;
        LQ_TRY(pool.make(c, &ev_panel));
        LQ_CUDA(c, cudaEventRecord(ev_panel, s_main));
        if (trace_blocks) btrace[blk].chain = ev_panel;
        if (pw) {
            // the next block's columns are complete once the aux stream has applied the last panel
            LQ_CUDA(c, cudaStreamWaitEvent(s_main, ev_aux_done, 0));
        } else {
            LQ_TRY(merge_block_t(G.as<double>()));
            if (nnext > 0) {
                if (ev_rest_prev) LQ_CUDA(c, cudaStreamWaitEvent(s_main, ev_rest_prev, 0));
                LQ_TRY(apply_block_reflector(c, Vb, ldv, Tblk, NB_OUT, true, mk, kb, Ctr, lda, nnext, W2.as<double>()));
            }
        }
        if (trace_blocks) {
            LQ_TRY(pool.make(c, &btrace[blk].next));
            LQ_CUDA(c, cudaEventRecord(btrace[blk].next, s_main));
        }
        {
            // the merged T: on its own stream right after the panels (so that it is ready when the side stream's
            // previous trailing update retires); then the side stream: trailing update beyond the next block, rhs
            cudaEvent_t ev_after;
            LQ_TRY(pool.make(c, &ev_after));
            if (pw) {
                StreamScope mg(c, s_merge);
                LQ_CUDA(c, cudaStreamWaitEvent(s_merge, ev_panel, 0));
                LQ_TRY(merge_block_t(Gmerge.as<double>()));
                LQ_CUDA(c, cudaEventRecord(ev_after, s_merge));
            } else {
                LQ_CUDA(c, cudaEventRecord(ev_after, s_main));  // T merged on the main stream
            }
            const int c_lo = k0 + kb + nnext;             // first column of the trailing update
            const int c_mid = std::max(c_lo, std::min(rsplit, npad));
            cudaEvent_t ev_left = nullptr, ev_right = nullptr;
            if (c_mid > c_lo) {
                StreamScope side(c, s_side);  // columns [c_lo, c_mid)
                LQ_CUDA(c, cudaStreamWaitEvent(s_side, ev_after, 0));
                LQ_TRY(apply_block_reflector(c, Vb, ldv, Tblk, NB_OUT, true, mk, kb, A + (size_t)k0 * lda + c_lo, lda, c_mid - c_lo,
                                             W2s.as<double>()));
                LQ_TRY(pool.make(c, &ev_left));
                LQ_CUDA(c, cudaEventRecord(ev_left, s_side));
                ev_rest_last[0] = ev_left;
            }
            {
                StreamScope side(c, s_side2);  // columns [c_mid, npad) and the right-hand sides
                LQ_CUDA(c, cudaStreamWaitEvent(s_side2, ev_after, 0));
                if (npad > c_mid)
                    LQ_TRY(apply_block_reflector(c, Vb, ldv, Tblk, NB_OUT, true, mk, kb, A + (size_t)k0 * lda + c_mid, lda, npad - c_mid,
                                                 W2s2.as<double>()));
                if (B && nrhs_pad > 0)
                    LQ_TRY(apply_block_reflector(c, Vb, ldv, Tblk, NB_OUT, true, mk, kb, B + (size_t)k0 * ldb, ldb, nrhs_pad,
                                                 W2s2.as<double>()));
                LQ_TRY(pool.make(c, &ev_right));
                LQ_CUDA(c, cudaEventRecord(ev_right, s_side2));
                ev_rest_last[1] = ev_right;
            }
            // the next block's columns of the NEXT iteration are the first columns of this trailing update
            ev_rest_prev = ev_left ? ev_left : ev_right;
            if (trace_blocks) btrace[blk].rest = ev_rest_prev;
        }
    }
    if (lookahead) {  // join
        for (cudaEvent_t e : ev_rest_last)
            if (e) LQ_CUDA(c, cudaStreamWaitEvent(s_main, e, 0));
    }
    if (trace_blocks) {
        LQ_CUDA(c, cudaStreamSynchronize(s_main));
        fprintf(stderr, "# blk  panels_done  chain_done  next_done  rest_done   (ms since start; m=%d npad=%d)\n", m, npad);
        for (int blk = 0; blk < nblocks; ++blk) {
            float t[4] = {-1.f, -1.f, -1.f, -1.f};
            cudaEvent_t evs[4] = {btrace[blk].panels, btrace[blk].chain, btrace[blk].next, btrace[blk].rest};
            for (int k = 0; k < 4; ++k)
                if (evs[k]) cudaEventElapsedTime(&t[k], ev_t0, evs[k]);
            fprintf(stderr, "%4d %10.3f %10.3f %10.3f %10.3f\n", blk, t[0], t[1], t[2], t[3]);
        }
    }
    return LQ_OK;
}

// back-substitution  R X = Y  for an upper-triangular R (n x n, ldr) and Y (n x k, ldy) in place.
// Small systems: one thread per right-hand side.
__global__ void __launch_bounds__(256) backsub_kernel(const double* __restrict__ R, int ldr, double* __restrict__ Y, int ldy,
                                                      int n, int k) {
    for (int col = blockIdx.x * blockDim.x + threadIdx.x; col < k; col += gridDim.x * blockDim.x) {
        for (int i = n - 1; i >= 0; --i) {
            double acc = Y[(long long)i * ldy + col];
            for (int cc = i + 1; cc < n; ++cc) acc = fma(-R[(long long)i * ldr + cc], Y[(long long)cc * ldy + col], acc);
            Y[(long long)i * ldy + col] = acc / R[(long long)i * ldr + i];
        }
    }
}
// One diagonal block (nb <= 128 rows) of a blocked back-substitution: Rbb in shared memory, CTA b solves a chunk
// of 32 right-hand sides; per row one divide, then a rank-1 update of the rows above by all threads.
__global__ void __launch_bounds__(256) backsub_diag_kernel(const double* __restrict__ R, int ldr, double* __restrict__ Y,
                                                           int ldy, int nb, int k) {
    extern __shared__ double bs_sm[];
    double* Rs = bs_sm;               // [nb][129]
    double* Ys = bs_sm + 128 * 129;   // [nb][33]
    __shared__ double xrow[32];
    const int c0 = blockIdx.x * 32, kc = min(32, k - c0);
    for (int e = threadIdx.x; e < nb * nb; e += 256) Rs[(e / nb) * 129 + e % nb] = R[(long long)(e / nb) * ldr + e % nb];
    for (int e = threadIdx.x; e < nb * 32; e += 256) {
        const int i = e >> 5, cc = e & 31;
        Ys[i * 33 + cc] = (cc < kc) ? Y[(long long)i * ldy + c0 + cc] : 0.0;
    }
    __syncthreads();
    for (int i = nb - 1; i >= 0; --i) {
        if (threadIdx.x < 32) {
            const double x = Ys[i * 33 + threadIdx.x] / Rs[i * 129 + i];
            xrow[threadIdx.x] = x;
            Ys[i * 33 + threadIdx.x] = x;
        }
        __syncthreads();
        for (int e = threadIdx.x; e < i * 32; e += 256) {
            const int r = e >> 5, cc = e & 31;
            Ys[r * 33 + cc] = fma(-Rs[r * 129 + i], xrow[cc], Ys[r * 33 + cc]);
        }
        __syncthreads();
    }
    for (int e = threadIdx.x; e < nb * 32; e += 256) {
        const int i = e >> 5, cc = e & 31;
        if (cc < kc) Y[(long long)i * ldy + c0 + cc] = Ys[i * 33 + cc];
    }
}
constexpr size_t BACKSUB_SMEM = (128 * 129 + 128 * 33) * sizeof(double);

// *info = 0, or 1 + the first j with R[j][j] exactly 0 (R: n x n, ldr); one CTA
__global__ void __launch_bounds__(256) singular_diag_kernel(const double* __restrict__ R, int ldr, int n, int* __restrict__ info) {
    __shared__ int first;
    if (threadIdx.x == 0) first = n;
    __syncthreads();
    for (int j = threadIdx.x; j < n; j += blockDim.x)
        if (R[(long long)j * ldr + j] == 0.0) atomicMin(&first, j);
    __syncthreads();
    if (threadIdx.x == 0) *info = (first < n) ? first + 1 : 0;
}

// R X = Y in place (Y: n x k, ldy; k even when the tensor-core GEMM is to be used for the off-diagonal part)
int back_substitute(Ctx* c, const double* R, int ldr, double* Y, int ldy, int n, int k) {
    if (n <= 256) return backsub_per_column(c, R, ldr, Y, ldy, n, k);
    const int nblk = (n + 127) / 128;
    for (int b = nblk - 1; b >= 0; --b) {
        const int r0 = b * 128, nb = std::min(128, n - r0), after = n - (r0 + nb);
        if (after > 0)  // Y_b -= R[b, after] X[after]
            LQ_TRY(gemm(c, false, false, nb, k, after, -1.0, R + (size_t)r0 * ldr + r0 + nb, ldr, Y + (size_t)(r0 + nb) * ldy, ldy,
                        1.0, Y + (size_t)r0 * ldy, ldy));
        LQ_TRY(launch<backsub_diag_kernel>(c, (k + 31) / 32, 256, BACKSUB_SMEM, c->stream, (int)BACKSUB_SMEM,
                                           R + (size_t)r0 * ldr + r0, ldr, Y + (size_t)r0 * ldy, ldy, nb, k));
    }
    return LQ_OK;
}

}  // namespace

int backsub_per_column(Ctx* c, const double* R, int ldr, double* Y, int ldy, int n, int k) {
    return launch<backsub_kernel>(c, std::max(1, (k + 255) / 256), 256, 0, c->stream, 0, R, ldr, Y, ldy, n, k);
}

int pad_columns(Ctx* c, const double* src, int lds, double* dst, int ldd, long long rows, int cols_src, int cols_dst) {
    return launch<pad_copy_kernel>(c, grid_for(c, rows * cols_dst), 256, 0, c->stream, 0, src, lds, dst, ldd, rows, cols_src,
                                   cols_dst);
}

int measure_max_cluster(Ctx* c) {
    constexpr auto kern = panel_cluster_kernel<4, 16>;
    LQ_TRY(set_attributes_once<kern>(c, 0, true));
    c->max_cluster = 1;
    for (int cs : {16, 8, 4, 2}) {
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3(cs);
        cfg.blockDim = dim3(PANEL_THREADS);
        cfg.dynamicSmemBytes = 0;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = cs;
        at[0].val.clusterDim.y = 1;
        at[0].val.clusterDim.z = 1;
        cfg.attrs = at;
        cfg.numAttrs = 1;
        int n = 0;
        cudaError_t e = cudaOccupancyMaxActiveClusters(&n, kern, &cfg);
        if (e == cudaSuccess && n >= 1) {
            c->max_cluster = cs;
            break;
        }
        cudaGetLastError();
    }
    return LQ_OK;
}

int blocked_householder_factor(Ctx* c, double* A, int lda, int m, int n, double* V, int ldv, double* B, int ldb,
                               int nrhs) {
    return factor_padded(c, A, lda, m, n, n, V, ldv, B, ldb, nrhs, nullptr);
}

int blocked_householder_qr(Ctx* c, const double* A, int m, int n, double* Q, double* R) {
    LQ_REQUIRE(c, m >= n && n >= 1, LQ_ERR_SHAPE, "householder_qr needs m >= n >= 1 (got %d x %d)", m, n);
    const int npad = (n + 31) / 32 * 32;
    DevBuf Aw, Vw, Qw;
    LQ_TRY(Aw.alloc(c, sizeof(double) * (size_t)m * npad));
    LQ_TRY(Vw.alloc(c, sizeof(double) * (size_t)m * npad));
    LQ_TRY(pad_columns(c, A, n, Aw.as<double>(), npad, m, n, npad));
    LQ_CUDA(c, cudaMemsetAsync(Vw.p, 0, sizeof(double) * (size_t)m * npad, c->stream));
    Factored keep;
    LQ_TRY(factor_padded(c, Aw.as<double>(), npad, m, npad, n, Vw.as<double>(), npad, nullptr, 0, 0, &keep));
    LQ_TRY(launch<extract_upper_kernel>(c, grid_for(c, (long long)n * n), 256, 0, c->stream, 0, Aw.as<double>(), npad, R, n));

    // ---- Q = H_0 H_1 ... H_{n-1} I  (thin, m x n), block reflectors applied in reverse order
    double* Qp = Q;
    int ldq = n;
    if (npad != n) {
        LQ_TRY(Qw.alloc(c, sizeof(double) * (size_t)m * npad));
        Qp = Qw.as<double>();
        ldq = npad;
    }
    // the A workspace is free now: reuse it for the scratch of the main stream (W2) and of the side stream (W)
    double* W = Aw.as<double>();
    double* W2 = W + (size_t)NB_OUT * npad;
    const bool ws_fits = (size_t)m * npad >= 2 * (size_t)NB_OUT * npad;
    DevBuf Wx;
    if (!ws_fits) {
        LQ_TRY(Wx.alloc(c, sizeof(double) * 2 * (size_t)NB_OUT * npad));
        W = Wx.as<double>();
        W2 = W + (size_t)NB_OUT * npad;
    }
    LQ_TRY(launch<set_identity_kernel>(c, grid_for(c, (long long)m * ldq), 256, 0, c->stream, 0, Qp, ldq, m, ldq));
    // A block reflector transforms every COLUMN of Q independently, so the columns are split into two contiguous
    // ranges that run the whole chain of applications on two streams with no synchronisation in between: the launch
    // gaps, split-K reductions and partial last waves of one range are filled by the other.  The split balances the
    // flops (block b touches the columns >= 128 b only): 3 s^2 - s^3 = 1  ->  s = 0.65.
    const bool two_ranges = ldq >= 2048 && ws_fits;
    const int split = two_ranges ? (int)(0.65 * ldq) / NB_OUT * NB_OUT : 0;
    cudaStream_t s_main = c->stream, s_side = c->lane[0];
    EventPool qpool;
    if (two_ranges) {
        cudaEvent_t e0;
        LQ_TRY(qpool.make(c, &e0));
        LQ_CUDA(c, cudaEventRecord(e0, s_main));
        LQ_CUDA(c, cudaStreamWaitEvent(s_side, e0, 0));
    }
    for (int blk = keep.nblocks - 1; blk >= 0; --blk) {
        const int k0 = blk * NB_OUT;
        const int kb = std::min(NB_OUT, npad - k0);
        const int mk = m - k0;
        if (mk <= 0) continue;
        const double* Vb = Vw.as<double>() + (size_t)k0 * npad + k0;
        const double* Tblk = keep.Tall.as<double>() + (size_t)blk * NB_OUT * NB_OUT;
        // only columns >= k0 of Q are touched by this block (Q[k0:, :k0] is still zero)
        const int c_hi = std::max(k0, split);  // main stream: columns [c_hi, ldq); side stream: [k0, split)
        LQ_TRY(apply_block_reflector(c, Vb, npad, Tblk, NB_OUT, false, mk, kb, Qp + (size_t)k0 * ldq + c_hi, ldq, ldq - c_hi, W2));
        if (k0 < split) {
            StreamScope side(c, s_side);
            LQ_TRY(apply_block_reflector(c, Vb, npad, Tblk, NB_OUT, false, mk, kb, Qp + (size_t)k0 * ldq + k0, ldq, split - k0, W));
        }
    }
    if (two_ranges) {
        cudaEvent_t e1;
        LQ_TRY(qpool.make(c, &e1));
        LQ_CUDA(c, cudaEventRecord(e1, s_side));
        LQ_CUDA(c, cudaStreamWaitEvent(s_main, e1, 0));
    }
    if (Qp != Q) return launch<unpad_copy_kernel>(c, grid_for(c, (long long)m * n), 256, 0, c->stream, 0, Qp, ldq, Q, n, m, n);
    return LQ_OK;
}

int large_lstsq_householder(Ctx* c, const double* A, const double* B, int m, int n, int nrhs, double* X, int* info) {
    LQ_REQUIRE(c, m >= n && n >= 1 && nrhs >= 1, LQ_ERR_SHAPE, "least squares needs m >= n >= 1, nrhs >= 1");
    const int npad = (n + 31) / 32 * 32;
    const int kpad = (nrhs + 1) / 2 * 2;
    DevBuf Aw, Vw, Bw;
    LQ_TRY(Aw.alloc(c, sizeof(double) * (size_t)m * npad));
    LQ_TRY(Vw.alloc(c, sizeof(double) * (size_t)m * npad));
    LQ_TRY(Bw.alloc(c, sizeof(double) * (size_t)m * kpad));
    LQ_TRY(pad_columns(c, A, n, Aw.as<double>(), npad, m, n, npad));
    LQ_TRY(pad_columns(c, B, nrhs, Bw.as<double>(), kpad, m, nrhs, kpad));
    LQ_CUDA(c, cudaMemsetAsync(Vw.p, 0, sizeof(double) * (size_t)m * npad, c->stream));
    LQ_TRY(factor_padded(c, Aw.as<double>(), npad, m, npad, n, Vw.as<double>(), npad, Bw.as<double>(), kpad, kpad, nullptr));
    if (info) LQ_TRY(launch<singular_diag_kernel>(c, 1, 256, 0, c->stream, 0, Aw.as<double>(), npad, n, info));
    LQ_TRY(back_substitute(c, Aw.as<double>(), npad, Bw.as<double>(), kpad, n, kpad));
    return launch<unpad_copy_kernel>(c, grid_for(c, (long long)n * nrhs), 256, 0, c->stream, 0, Bw.as<double>(), kpad, X, nrhs, n,
                                     nrhs);
}

}  // namespace lq

using namespace lq;

extern "C" {

// diagnostics: one panel factorisation (mp x nb at A, lda) with an explicit kernel version (see panel_factor_v)
int lq_debug_panel(lq_ctx* h, double* A, int lda, double* V, int ldv, double* T, int ldt, int mp, int nb, int version) {
    Ctx* c = as_ctx(h);
    if (!c) return LQ_ERR_ARG;
    LQ_REQUIRE(c, version == 0 || version == 1 || version == 3, LQ_ERR_ARG,
               "debug_panel: panel kernel version %d does not exist (0, 1 and 3 do)", version);
    LQ_CUDA(c, cudaSetDevice(c->device));
    return panel_factor_v(c, A, lda, V, ldv, T, ldt, mp, nb, version);
}

// diagnostics: the 256-rows-per-CTA st.async panel kernel with clock64() stamps (2 warps x 32 columns x 8 phases)
int lq_debug_panel_trace(lq_ctx* h, double* A, int lda, double* V, int ldv, double* T, int ldt, int mp, long long* trace) {
    Ctx* c = as_ctx(h);
    if (!c) return LQ_ERR_ARG;
    LQ_CUDA(c, cudaSetDevice(c->device));
    LQ_REQUIRE(c, mp <= c->max_cluster * Panel2Cfg<8>::ROWS_PER_CTA, LQ_ERR_SHAPE, "panel too tall for the traced kernel");
    if (mp <= Panel2Cfg<8>::ROWS_PER_CTA)  // the one-CTA kernel's stamps
        return launch<panel2_cluster_kernel<8, true, true>>(c, 1, P2_THREADS, 0, c->stream, 0, A, lda, V, ldv, T, ldt, mp, trace);
    int cs = 1;
    while (cs * Panel2Cfg<8>::ROWS_PER_CTA < mp) cs *= 2;
    return launch_cluster<panel2_cluster_kernel<8, true>>(c, cs, P2_THREADS, A, lda, V, ldv, T, ldt, mp, trace);
}

int lq_householder_qr_dev(lq_ctx* h, const double* A, int m, int n, double* Q, double* R) {
    Ctx* c = as_ctx(h);
    if (!c) return LQ_ERR_ARG;
    LQ_REQUIRE(c, m >= 1 && n >= 1 && m >= n, LQ_ERR_SHAPE, "householder_qr needs m >= n >= 1 (got %d x %d)", m, n);
    LQ_CUDA(c, cudaSetDevice(c->device));
    // small problems: the one-CTA shared-memory kernel (a single launch)
    if ((size_t)m * n <= 4096) return hh_qr_batched_stream(c, c->stream, A, 1, m, n, Q, R, false);
    // launch-latency-bound sizes: replay the whole multi-stream schedule as one CUDA graph (second call with the same
    // shape and buffers captures it, later calls replay it).  Measured (tools/check_graph.py): 256^2 0.78 -> 0.67 ms,
    // 1000^2 3.51 -> 2.99, 2048^2 6.32 -> 5.65, 4096^2 15.9 -> 14.7, 8192^2 62.1 -> 60.5.  The graph is instantiated with
    // cudaGraphInstantiateFlagUseNodePriority: without the captured stream priorities (panel chain ahead of the bulk
    // updates) the 8192^2 replay is 5 % SLOWER than the plain launches (65.4 ms).
    if (c->env_no_graph || (size_t)m * n > ((size_t)1 << 26)) return blocked_householder_qr(c, A, m, n, Q, R);
    Ctx::GraphEntry* e = nullptr;
    for (auto& g : c->graphs)
        if (g.m == m && g.n == n && g.A == A && g.Q == Q && g.R == R) e = &g;
    if (!e) {
        // a graph keeps its scratch allocations (4 matrix-sized buffers) alive: at most one cached graph of a large shape
        if ((size_t)m * n > ((size_t)1 << 22)) {
            for (size_t i = 0; i < c->graphs.size();) {
                if ((size_t)c->graphs[i].m * c->graphs[i].n > ((size_t)1 << 22)) {
                    if (c->graphs[i].exec) cudaGraphExecDestroy(c->graphs[i].exec);
                    c->graphs.erase(c->graphs.begin() + i);
                } else {
                    ++i;
                }
            }
        }
        if (c->graphs.size() >= 8) {  // evict the least recently used entry
            size_t lru = 0;
            for (size_t i = 1; i < c->graphs.size(); ++i)
                if (c->graphs[i].stamp < c->graphs[lru].stamp) lru = i;
            if (c->graphs[lru].exec) cudaGraphExecDestroy(c->graphs[lru].exec);
            c->graphs.erase(c->graphs.begin() + lru);
        }
        Ctx::GraphEntry ne;
        ne.m = m, ne.n = n, ne.A = A, ne.Q = Q, ne.R = R, ne.stamp = ++c->graph_clock;
        c->graphs.push_back(ne);
        return blocked_householder_qr(c, A, m, n, Q, R);  // warm-up call: plain launches
    }
    e->stamp = ++c->graph_clock;
    if (e->state == 1) {
        LQ_CUDA(c, cudaGraphLaunch(e->exec, c->stream));
        c->launches += e->launches;
        return LQ_OK;
    }
    if (e->state < 0) return blocked_householder_qr(c, A, m, n, Q, R);
    // capture (the side streams join the capture through the events they wait for, and are joined back by the schedule)
    const long long l0 = c->launches;
    cudaGraph_t graph = nullptr;
    if (cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
        cudaGetLastError();
        e->state = -1;
        return blocked_householder_qr(c, A, m, n, Q, R);
    }
    const int rc = blocked_householder_qr(c, A, m, n, Q, R);
    const cudaError_t ce = cudaStreamEndCapture(c->stream, &graph);
    cudaGraphExec_t exec = nullptr;
    if (rc == LQ_OK && ce == cudaSuccess && graph && cudaGraphInstantiateWithFlags(&exec, graph, cudaGraphInstantiateFlagUseNodePriority) == cudaSuccess) {
        e->exec = exec;
        e->launches = c->launches - l0;
        e->state = 1;
        cudaGraphDestroy(graph);
        LQ_CUDA(c, cudaGraphLaunch(e->exec, c->stream));
        return LQ_OK;
    }
    // not capturable (e.g. unjoined side stream for this shape): remember, clear the sticky capture error, run plainly
    if (graph) cudaGraphDestroy(graph);
    cudaGetLastError();
    e->state = -1;
    c->launches = l0;
    return blocked_householder_qr(c, A, m, n, Q, R);
}

}  // extern "C"

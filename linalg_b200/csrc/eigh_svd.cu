// Gram matrix, symmetric eigen-solver and economy SVD through the A^T A route (linalg/svd.py:10-82): the two-sided and
// one-sided Jacobi kernels with their eigenvector, eigenvalue and sort kernels, the SVD post-processing, and the orthonormal
// completion of U with its counter-based (Philox) candidate generator.
#include "../../include/linalg_b200.h"
#include "ops.cuh"

namespace lq {

namespace {

// ------------------------------------------------------------------ Jacobi eigen-solver
// Two-sided cyclic Jacobi with the round-robin ("circle") parallel ordering.  One CTA owns the
// matrix (shared memory when it fits, global memory otherwise); every round applies n/2 disjoint
// rotations, first to the columns then to the rows.  The (c, s) pairs are logged so that the
// eigenvectors can be accumulated afterwards by independent CTAs (one row of V each).  Pairs of a round: rr_pair
// (common.cuh).

__global__ void __launch_bounds__(1024) jacobi_kernel(const double* __restrict__ G, int n, double* __restrict__ Awork,
                                                     int use_global, double2* __restrict__ rotlog, int max_sweeps, double rel_tol,
                                                     int* __restrict__ nrounds_out, double* __restrict__ lambda) {
    extern __shared__ __align__(16) double sm[];
    const int ne = (n + 1) & ~1;          // padded to even; the pad index never rotates (zero coupling)
    const int ld = ne | 1;                // odd pitch
    double* Am = use_global ? Awork : sm;
    double2* cs = reinterpret_cast<double2*>(use_global ? sm : sm + (size_t)ne * ld + (ne & 1 ? 1 : 0) + 1);
    // align cs to 16 bytes
    cs = reinterpret_cast<double2*>((reinterpret_cast<uintptr_t>(cs) + 15) & ~(uintptr_t)15);
    __shared__ int s_rot, s_exp;
    __shared__ double s_scale;
    __shared__ int2 pq[1024];  // pairs of the current round (n <= 2048)
    const int tid = threadIdx.x, nt = blockDim.x;
    const int half = ne / 2;

    int bad = 0;
    for (int e = tid; e < ne * ne; e += nt) {
        const int i = e / ne, j = e - i * ne;
        const double v = (i < n && j < n) ? G[(size_t)i * n + j] : 0.0;
        bad |= !isfinite(v);
        Am[(size_t)i * ld + j] = v;
    }
    // A NaN or infinite entry: no rotation test can be evaluated on it (an infinite diagonal makes floor_abs infinite and
    // stops every rotation, a NaN pair never rotates), so the diagonal left behind would be finite values that are not
    // eigenvalues.  Every eigenvalue is NaN instead and no sweep runs (V = I, written in full by the replay).
    const int nonfinite = __syncthreads_or(bad);
    // work on 2^-e G with max|diag| in [1, 2): the rotation test forms app * aqq, which would overflow from max|diag| ~ 2^512.
    // The scaling is exact; lambda is scaled back by 2^e below.
    if (tid == 0) {
        double g = 0.0;
        for (int i = 0; i < n; ++i) g = fmax(g, fabs(Am[(size_t)i * ld + i]));
        const int e = (g > 0.0 && isfinite(g)) ? ilogb(g) : 0;
        s_exp = e;
        s_scale = scalbn(g, -e);
    }
    __syncthreads();
    const int gexp = s_exp;
    if (gexp != 0)
        for (int e = tid; e < ne * ne; e += nt) {
            double* a = Am + (size_t)(e / ne) * ld + e % ne;
            *a = scalbn(*a, -gexp);
        }
    __syncthreads();
    const double floor_abs = 4.9303806576313238e-32 * s_scale;  // eps^2 * max|diag|

    int rounds = 0;
    for (int sweep = 0; sweep < (nonfinite ? 0 : max_sweeps); ++sweep) {
        if (tid == 0) s_rot = 0;
        __syncthreads();
        for (int rd = 0; rd < ne - 1; ++rd, ++rounds) {
            // rotation parameters of this round
            for (int kk = tid; kk < half; kk += nt) {
                int p, q;
                rr_pair(ne, rd, kk, p, q);
                pq[kk] = make_int2(p, q);
                const double app = Am[(size_t)p * ld + p], aqq = Am[(size_t)q * ld + q], apq = Am[(size_t)p * ld + q];
                double cc = 1.0, ss = 0.0;
                if (fabs(apq) > floor_abs && fabs(apq) > rel_tol * sqrt(fabs(app * aqq))) {
                    const double tau = (aqq - app) / (2.0 * apq);
                    const double t = copysign(1.0, tau) / (fabs(tau) + sqrt(1.0 + tau * tau));
                    cc = 1.0 / sqrt(1.0 + t * t);
                    ss = t * cc;
                    s_rot = 1;  // benign race: every writer stores the same value (a same-address atomic serialises 64 lanes)
                }
                cs[kk] = make_double2(cc, ss);
                rotlog[(size_t)rounds * half + kk] = make_double2(cc, ss);
            }
            __syncthreads();
            // columns: A[:, p], A[:, q] -- one warp per rotation pair, lanes over the rows; 32-bit indexing and a
            // 4-way unrolled body (the solver is instruction bound on its single SM)
            const int wid = tid >> 5, ln = tid & 31, nwp = nt >> 5;
            for (int k = wid; k < half; k += nwp) {
                const int p = pq[k].x, q = pq[k].y;
                const double2 r2 = cs[k];
                if (r2.y != 0.0) {
                    double* colp = Am + p;
                    double* colq = Am + q;
                    int i = ln;
                    for (; i + 96 < ne; i += 128) {
                        double ap[4], aq[4];
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            ap[u] = colp[(i + 32 * u) * ld];
                            aq[u] = colq[(i + 32 * u) * ld];
                        }
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            colp[(i + 32 * u) * ld] = r2.x * ap[u] - r2.y * aq[u];
                            colq[(i + 32 * u) * ld] = r2.y * ap[u] + r2.x * aq[u];
                        }
                    }
                    for (; i < ne; i += 32) {
                        const double ap = colp[i * ld], aq = colq[i * ld];
                        colp[i * ld] = r2.x * ap - r2.y * aq;
                        colq[i * ld] = r2.y * ap + r2.x * aq;
                    }
                }
            }
            __syncthreads();
            // rows: A[p, :], A[q, :]
            for (int k = wid; k < half; k += nwp) {
                const int p = pq[k].x, q = pq[k].y;
                const double2 r2 = cs[k];
                if (r2.y != 0.0) {
                    double* rowp = Am + p * ld;
                    double* rowq = Am + q * ld;
                    int j = ln;
                    for (; j + 96 < ne; j += 128) {
                        double ap[4], aq[4];
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            ap[u] = rowp[j + 32 * u];
                            aq[u] = rowq[j + 32 * u];
                        }
#pragma unroll
                        for (int u = 0; u < 4; ++u) {
                            rowp[j + 32 * u] = r2.x * ap[u] - r2.y * aq[u];
                            rowq[j + 32 * u] = r2.y * ap[u] + r2.x * aq[u];
                        }
                    }
                    for (; j < ne; j += 32) {
                        const double ap = rowp[j], aq = rowq[j];
                        rowp[j] = r2.x * ap - r2.y * aq;
                        rowq[j] = r2.y * ap + r2.x * aq;
                    }
                }
            }
            __syncthreads();
        }
        const int nrot = s_rot;
        __syncthreads();
        if (nrot == 0) break;
    }
    if (tid == 0) *nrounds_out = rounds;
    for (int i = tid; i < n; i += nt) lambda[i] = nonfinite ? eig_nan() : scalbn(Am[(size_t)i * ld + i], gexp);
}


// One-sided (Hestenes) Jacobi for n <= 128: the columns of B = G J_1 J_2 ... are rotated until they are mutually
// orthogonal, then B = V diag(lambda).  Why it is faster than jacobi_kernel: a round of the two-sided kernel reads and
// writes the whole matrix twice (rows and columns: 98 k doubles of shared-memory traffic at n = 128, the 128 B/clk
// port is the limit) behind three block barriers; here a round touches every column once and the three inner
// products of a pair stay in registers.  Eight lanes own a column pair (16-byte loads, two rows per lane, 16-row
// stride), four pairs per warp, Newton-refined MUFU reciprocals / rsqrt instead of the IEEE subroutines.
//
// Ordering (block round-robin): the ne / 4 blocks of four columns play a round-robin tournament; in a super-round a
// warp owns one block pair (X, Y) and works through its 4 x 4 cross pairs in four steps that need only __syncwarp
// (group g keeps column x_g in registers and meets y_{(g + t) mod 4} in step t), so the block barrier comes once per
// FOUR rounds and the warps drift apart inside a super-round: loads, FP64 and the scalar chains of different warps
// overlap instead of marching in lock step.  The six pairs inside each block are done in three steps at the start of
// a sweep.  One sweep = 3 + 4 (ne / 4 - 1) steps of ne / 2 disjoint pairs = every pair once.  The (c, s) log is
// indexed [step][slot = 4 warp + group] (64 slots per step); jacobi1s_pair() maps it back to the columns for the eigenvector replay.
// ne = n padded to a multiple of 16 (zero columns never rotate).  B is left in Bout (column-major, pitch ne).
__host__ __device__ inline int jacobi1s_steps_per_sweep(int ne) { return 3 + 4 * (ne / 4 - 1); }
__device__ __forceinline__ bool jacobi1s_pair(int ne, int step, int slot, int& p, int& q) {
    const int nblk = ne >> 2, w = slot >> 2, g = slot & 3;
    if (step < 3) {
        const int b = w + 16 * (g >> 1);  // two blocks per warp
        if (b >= nblk) return false;
        const int gg = g & 1;
        // step 0: (0,1) (2,3); step 1: (0,2) (1,3); step 2: (0,3) (1,2)
        const int lo = (gg == 0) ? 0 : (step == 0 ? 2 : 1);
        const int hi = (gg == 0) ? (step + 1) : (step == 0 ? 3 : (step == 1 ? 3 : 2));
        p = 4 * b + lo;
        q = 4 * b + hi;
        return true;
    }
    if (w >= (nblk >> 1)) return false;
    const int sr = (step - 3) >> 2, t = (step - 3) & 3;
    int X, Y;
    rr_pair(nblk, sr, w, X, Y);
    p = 4 * X + g;
    q = 4 * Y + ((g + t) & 3);
    return true;
}

// one rotation of the column pair held by an 8-lane group: ap / aq are the group's rows of columns p and q
template <int NUMAX>
__device__ __forceinline__ void jacobi1s_rotate(double (&ap)[2 * NUMAX], double (&aq)[2 * NUMAX], int NU, bool active, double floor_abs,
                                                double rel_tol, double& cc, double& ss) {
    double a0 = 0.0, a1 = 0.0, b0 = 0.0, b1 = 0.0, g0 = 0.0, g1 = 0.0;
#pragma unroll
    for (int u = 0; u < NUMAX; ++u) {
        if (u < NU) {
            a0 = fma(ap[2 * u], ap[2 * u], a0), a1 = fma(ap[2 * u + 1], ap[2 * u + 1], a1);
            b0 = fma(aq[2 * u], aq[2 * u], b0), b1 = fma(aq[2 * u + 1], aq[2 * u + 1], b1);
            g0 = fma(ap[2 * u], aq[2 * u], g0), g1 = fma(ap[2 * u + 1], aq[2 * u + 1], g1);
        }
    }
    double alpha = a0 + a1, beta = b0 + b1, gamma = g0 + g1;
#pragma unroll
    for (int o = 1; o < 8; o <<= 1) {
        alpha += __shfl_xor_sync(0xffffffffu, alpha, o);
        beta += __shfl_xor_sync(0xffffffffu, beta, o);
        gamma += __shfl_xor_sync(0xffffffffu, gamma, o);
    }
    cc = 1.0;
    ss = 0.0;
    // rotate while |p.q| > rel_tol ||p|| ||q||   (squared: gamma^2 > rel_tol^2 alpha beta)
    if (active && fabs(gamma) > floor_abs && gamma * gamma > rel_tol * rel_tol * (alpha * beta)) {
        // zeta = (beta - alpha) / (2 gamma), t = sign(zeta) / (|zeta| + sqrt(1 + zeta^2)), c = 1 / sqrt(1 + t^2)
        double zeta = (beta - alpha) * (0.5 * rcp_nr_t<2>(gamma));
        zeta = fmin(fmax(zeta, -1e100), 1e100);
        const double w = fma(zeta, zeta, 1.0);
        const double sq = w * rsqrt_nr_t<2>(w);
        const double t = copysign(rcp_nr_t<2>(fabs(zeta) + sq), zeta);
        cc = rsqrt_nr_t<2>(fma(t, t, 1.0));
        ss = t * cc;
#pragma unroll
        for (int u = 0; u < 2 * NUMAX; ++u) {
            if (u < 2 * NU) {
                const double x = ap[u], y = aq[u];
                ap[u] = cc * x - ss * y;
                aq[u] = ss * x + cc * y;
            }
        }
    }
}

template <int NU_T>  // NU_T = 8: the n = 128 specialisation (no row guards); 0: ne / 16 at run time
__global__ void __launch_bounds__(512) jacobi1s_kernel(const double* __restrict__ G, int n, int ne, double2* __restrict__ rotlog,
                                                       int max_sweeps, double rel_tol, int* __restrict__ nsteps_out,
                                                       double* __restrict__ Bout, unsigned short* __restrict__ pairtab,
                                                       double* __restrict__ colnorm, int allow_direct) {
    constexpr int NUMAX = 8;
    extern __shared__ __align__(16) double Bm[];  // ne x ne, column-major
    __shared__ int s_rot, s_exp;
    __shared__ double s_scale;
    const int tid = threadIdx.x, nt = blockDim.x;
    const int wid = tid >> 5, ln = tid & 31, g = ln >> 3, r8 = ln & 7;
    const int NU = NU_T ? NU_T : ne / 16, nblk = ne / 4;
    const int slot = 4 * wid + g;

    int bad = 0;
    for (int e = tid; e < ne * ne; e += nt) {
        const int j = e / ne, i = e - j * ne;
        const double v = (i < n && j < n) ? G[(size_t)j * n + i] : 0.0;  // G is symmetric: read it row-wise
        bad |= !isfinite(v);
        Bm[e] = v;
    }
    // a NaN or infinite entry: no sweep, the replay gives V = I and eig_rayleigh_kernel writes NaN for every eigenvalue
    // (nsteps_out[3]); see jacobi_kernel
    const int nonfinite = __syncthreads_or(bad);
    if (tid == 0) nsteps_out[3] = nonfinite;
    // B = 2^-e G with max|diag| in [1, 2): the rotation test multiplies four entries (alpha beta, gamma^2), which would
    // overflow from max|diag| ~ 2^256 and underflow below ~ 2^-256.  The scaling is exact; eig_rayleigh_kernel scales
    // lambda back by 2^e (nsteps_out[2]).
    if (tid == 0) {
        double gmax = 0.0;
        for (int i = 0; i < n; ++i) gmax = fmax(gmax, fabs(Bm[i * ne + i]));
        const int e = (gmax > 0.0 && isfinite(gmax)) ? ilogb(gmax) : 0;
        s_exp = e;
        s_scale = scalbn(gmax, -e);
        nsteps_out[2] = e;
    }
    __syncthreads();
    if (s_exp != 0)
        for (int e = tid; e < ne * ne; e += nt) Bm[e] = scalbn(Bm[e], -s_exp);
    __syncthreads();
    const double floor_abs = 4.9303806576313238e-32 * s_scale * s_scale;  // (eps * max|diag|)^2
    // the pair schedule of one sweep for the eigenvector replay: p | q << 8, 0xffff = idle slot
    for (int e = tid; e < jacobi1s_steps_per_sweep(ne) * 64; e += nt) {
        int p, q;
        pairtab[e] = jacobi1s_pair(ne, e >> 6, e & 63, p, q) ? (unsigned short)(p | (q << 8)) : (unsigned short)0xffff;
    }

    auto load_col = [&](int col, double (&a)[2 * NUMAX]) {
        const double* cp = Bm + col * ne + 2 * r8;
#pragma unroll
        for (int u = 0; u < NUMAX; ++u)
            if (u < NU) {
                const double2 x = *reinterpret_cast<const double2*>(cp + 16 * u);
                a[2 * u] = x.x, a[2 * u + 1] = x.y;
            }
    };
    auto store_col = [&](int col, const double (&a)[2 * NUMAX]) {
        double* cp = Bm + col * ne + 2 * r8;
#pragma unroll
        for (int u = 0; u < NUMAX; ++u)
            if (u < NU) *reinterpret_cast<double2*>(cp + 16 * u) = make_double2(a[2 * u], a[2 * u + 1]);
    };

    int step_base = 0;
    const int sps = jacobi1s_steps_per_sweep(ne);
    int rotated = 0;
    for (int sweep = 0; sweep < (nonfinite ? 0 : max_sweeps); ++sweep, step_base += sps) {
        if (tid == 0) s_rot = 0;
        rotated = 0;
        // ---- the pairs inside the blocks
#pragma unroll 1
        for (int st = 0; st < 3; ++st) {
            int p = 0, q = 0;
            const bool active = jacobi1s_pair(ne, st, slot, p, q);
            double ap[2 * NUMAX], aq[2 * NUMAX], cc, ss;
            load_col(p, ap);
            load_col(q, aq);
            jacobi1s_rotate<NUMAX>(ap, aq, NU, active, floor_abs, rel_tol, cc, ss);
            if (ss != 0.0) {
                store_col(p, ap);
                store_col(q, aq);
                rotated = 1;
            }
            if (r8 == 0) rotlog[(size_t)(step_base + st) * 64 + slot] = make_double2(cc, ss);
            __syncwarp();
        }
        __syncthreads();
        // ---- block round-robin
#pragma unroll 1
        for (int sr = 0; sr < nblk - 1; ++sr) {
            int p = 0, q = 0;
            const bool active = jacobi1s_pair(ne, 3 + 4 * sr, slot, p, q);
            const int qb = q - (g & 3);  // first column of block Y
            double ap[2 * NUMAX], aq[2 * NUMAX], cc, ss;
            load_col(p, ap);
            bool xdirty = false;
#pragma unroll 1
            for (int t = 0; t < 4; ++t) {
                const int qq = active ? qb + ((g + t) & 3) : 0;
                load_col(qq, aq);
                jacobi1s_rotate<NUMAX>(ap, aq, NU, active, floor_abs, rel_tol, cc, ss);
                if (ss != 0.0) {
                    store_col(qq, aq);
                    xdirty = true;
                }
                if (r8 == 0) rotlog[(size_t)(step_base + 3 + 4 * sr + t) * 64 + slot] = make_double2(cc, ss);
                __syncwarp();
            }
            if (xdirty) {
                store_col(p, ap);
                rotated = 1;
            }
            __syncthreads();
        }
        if (rotated) s_rot = 1;  // benign race: every writer stores the same value
        __syncthreads();
        const int nrot = s_rot;
        __syncthreads();
        if (nrot == 0) {
            step_base += sps;
            break;
        }
    }
    if (tid == 0) *nsteps_out = step_base;
    for (int e = tid; e < ne * ne; e += nt) Bout[e] = Bm[e];
    // The converged columns are b_i = G v_i = lambda_i v_i: for a well-conditioned PSD matrix the eigenvectors are simply the
    // normalised columns (error ~ eps lambda_max / lambda_i), and the replay of the rotation log (0.22 ms at n = 128) can be
    // skipped.  nsteps_out[1] = 1 tells the two follow-up kernels to take that route (lambda_min > 1e-2 lambda_max: vectors to ~1e-14).
    __shared__ double s_cn[128];
    for (int col = tid >> 3; col < ne; col += nt >> 3) {
        double a[2 * NUMAX];
        load_col(col, a);
        double n0 = 0.0, n1 = 0.0;
#pragma unroll
        for (int u = 0; u < NUMAX; ++u)
            if (u < NU) n0 = fma(a[2 * u], a[2 * u], n0), n1 = fma(a[2 * u + 1], a[2 * u + 1], n1);
        double nn = n0 + n1;
#pragma unroll
        for (int o = 1; o < 8; o <<= 1) nn += __shfl_xor_sync(0xffffffffu, nn, o);
        if (r8 == 0) s_cn[col] = sqrt(nn);
    }
    __syncthreads();
    for (int i = tid; i < n; i += nt) colnorm[i] = s_cn[i];
    if (tid == 0) {
        double mn = 1e300, mx = 0.0;
        for (int i = 0; i < n; ++i) mn = fmin(mn, s_cn[i]), mx = fmax(mx, s_cn[i]);
        nsteps_out[1] = (allow_direct && !nonfinite && mx > 0.0 && mn > 1e-2 * mx) ? 1 : 0;
    }
}

// V[:, i] = b_i / ||b_i|| when the Jacobi kernel found the matrix well conditioned (see there); V row-major n x n
__global__ void __launch_bounds__(256) eigvec_from_b_kernel(const double* __restrict__ B, int ne, const double* __restrict__ colnorm,
                                                            const int* __restrict__ flags, int n, double* __restrict__ V) {
    if (flags[1] == 0) return;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n * n; e += gridDim.x * blockDim.x) {
        const int j = e / n, i = e - j * n;  // V[j][i] = B[row j of column i]
        V[e] = B[(size_t)i * ne + j] / colnorm[i];
    }
}

// V = J_1 J_2 ... for the one-sided kernel's log: one WARP per row of V (the row lives in warp-private shared memory,
// a step's ne / 2 rotations are disjoint: two slots per lane, one __syncwarp per step)
__global__ void __launch_bounds__(128) jacobi1s_apply_kernel(const double2* __restrict__ rotlog, const int* __restrict__ nsteps,
                                                            const unsigned short* __restrict__ pairtab, int n, int ne,
                                                            double* __restrict__ V) {
    __shared__ double rows[4][128];
    const int wid = threadIdx.x >> 5, ln = threadIdx.x & 31;
    const int b = blockIdx.x * 4 + wid;
    if (b >= n || nsteps[1] != 0) return;  // (well-conditioned matrix: the eigenvectors come straight from B)
    double* row = rows[wid];
    for (int j = ln; j < ne; j += 32) row[j] = (j == b) ? 1.0 : 0.0;
    __syncwarp();
    const int sps = jacobi1s_steps_per_sweep(ne);
    const int S = *nsteps;
    // the log lives in L2: fetch DEPTH steps at a time (rotations and pair schedule), then apply them, so that one L2
    // round trip is paid per DEPTH steps
    constexpr int DEPTH = 8;
    int sst = 0;
    for (int st0 = 0; st0 < S; st0 += DEPTH) {
        double2 cs0[DEPTH], cs1[DEPTH];
        unsigned pq0[DEPTH], pq1[DEPTH];
#pragma unroll
        for (int d = 0; d < DEPTH; ++d) {
            cs0[d] = cs1[d] = make_double2(1.0, 0.0);
            pq0[d] = pq1[d] = 0xffff;
            if (st0 + d < S) {
                int sd = sst + d;
                sd = sd >= sps ? sd - sps : sd;
                cs0[d] = rotlog[(size_t)(st0 + d) * 64 + ln];
                cs1[d] = rotlog[(size_t)(st0 + d) * 64 + ln + 32];
                pq0[d] = pairtab[sd * 64 + ln];
                pq1[d] = pairtab[sd * 64 + ln + 32];
            }
        }
        sst += DEPTH;
        sst = sst >= sps ? sst - sps : sst;
#pragma unroll
        for (int d = 0; d < DEPTH; ++d) {
            if (cs0[d].y != 0.0 && pq0[d] != 0xffff) {
                const int p = pq0[d] & 255, q = pq0[d] >> 8;
                const double vp = row[p], vq = row[q];
                row[p] = cs0[d].x * vp - cs0[d].y * vq;
                row[q] = cs0[d].y * vp + cs0[d].x * vq;
            }
            if (cs1[d].y != 0.0 && pq1[d] != 0xffff) {
                const int p = pq1[d] & 255, q = pq1[d] >> 8;
                const double vp = row[p], vq = row[q];
                row[p] = cs1[d].x * vp - cs1[d].y * vq;
                row[q] = cs1[d].y * vp + cs1[d].x * vq;
            }
            __syncwarp();
        }
    }
    for (int j = ln; j < n; j += 32) V[(size_t)b * n + j] = row[j];
}

// lambda_i = 2^e v_i^T (2^-e G v_i) = 2^e v_i . b_i   (B = 2^-e G V column-major with pitch ne, e = flags[2]; V row-major
// n x n, eigenvectors in columns); NaN for a non-finite G (flags[3])
__global__ void __launch_bounds__(256) eig_rayleigh_kernel(const double* __restrict__ B, int ne, const double* __restrict__ V, int n,
                                                           const int* __restrict__ flags, double* __restrict__ lambda) {
    const int wid = threadIdx.x >> 5, ln = threadIdx.x & 31;
    const int e = flags[2], nonfinite = flags[3];
    for (int i = blockIdx.x * (blockDim.x >> 5) + wid; i < n; i += gridDim.x * (blockDim.x >> 5)) {
        double acc = 0.0;
        for (int j = ln; j < n; j += 32) acc = fma(V[(size_t)j * n + i], B[(size_t)i * ne + j], acc);
        acc = warp_sum(acc);
        if (ln == 0) lambda[i] = nonfinite ? eig_nan() : scalbn(acc, e);
    }
}

// V = J_1 J_2 ... (rows of the identity transformed independently): CTA b owns row b of V.
__global__ void __launch_bounds__(256) jacobi_apply_kernel(const double2* __restrict__ rotlog, const int* __restrict__ nrounds,
                                                           int n, int ne, double* __restrict__ V) {
    extern __shared__ double row[];
    const int half = ne / 2;
    const int b = blockIdx.x;
    for (int j = threadIdx.x; j < ne; j += blockDim.x) row[j] = (j == b) ? 1.0 : 0.0;
    __syncthreads();
    const int R = *nrounds;
    // a round's ne / 2 rotations are disjoint: the threads of the CTA share them (any ne / 2, not just <= blockDim.x)
    for (int rd = 0; rd < R; ++rd) {
        for (int k = threadIdx.x; k < half; k += blockDim.x) {
            const double2 cur = rotlog[(size_t)rd * half + k];
            if (cur.y != 0.0) {
                int p, q;
                rr_pair(ne, rd % (ne - 1), k, p, q);
                const double vp = row[p], vq = row[q];
                row[p] = cur.x * vp - cur.y * vq;
                row[q] = cur.y * vp + cur.x * vq;
            }
        }
        __syncthreads();
    }
    for (int j = threadIdx.x; j < n; j += blockDim.x) V[(size_t)b * n + j] = row[j];
}

// sort eigenvalues descending (rank by counting), permute the columns of V accordingly.  Any number of CTAs: every CTA
// ranks all eigenvalues itself (n^2 compares) and moves its slice of V (one CTA took 35 us at n = 128).  The order is
// eig_desc_before's (NaN first), so the ranks are a permutation and every slot of lam_out and of V is written for any input.
__global__ void __launch_bounds__(256) eig_sort_kernel(const double* __restrict__ lam_in, const double* __restrict__ Vin, int n,
                                                       double* __restrict__ lam_out, double* __restrict__ Vout) {
    extern __shared__ int rank_of[];
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const double li = lam_in[i];
        int rk = 0;
        for (int j = 0; j < n; ++j) rk += eig_desc_before(lam_in[j], j, li, i);
        rank_of[i] = rk;
        if (blockIdx.x == 0) lam_out[rk] = li;
    }
    __syncthreads();
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n * n; e += gridDim.x * blockDim.x) {
        const int r = e / n, cidx = e - r * n;
        Vout[(size_t)r * n + rank_of[cidx]] = Vin[e];
    }
}

// s = sqrt(max(lambda, 0)) (NaN stays NaN); M2 = V diag(1/s for s > tol else 0); Vt = V^T; rank = #(s > tol).  Any number
// of CTAs (one CTA spent 48 us on 16 384 square roots and divisions at n = 128): the singular values are formed once per CTA
// in shared memory.
__global__ void __launch_bounds__(256) svd_post_kernel(const double* __restrict__ lam, const double* __restrict__ V, int n,
                                                       double tol, double* __restrict__ s, double* __restrict__ M2,
                                                       double* __restrict__ Vt, int* __restrict__ rank) {
    extern __shared__ double sv[];
    __shared__ int cnt;
    if (threadIdx.x == 0) cnt = 0;
    __syncthreads();
    for (int j = threadIdx.x; j < n; j += blockDim.x) {
        const double sj = sqrt_clip0(lam[j]);
        sv[j] = sj;
        if (blockIdx.x == 0) {
            s[j] = sj;
            if (sj > tol) atomicAdd(&cnt, 1);
        }
    }
    __syncthreads();
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n * n; e += gridDim.x * blockDim.x) {
        const int i = e / n, j = e - i * n;
        const double sj = sv[j];
        const double v = V[e];
        M2[e] = (sj > tol) ? v / sj : 0.0;
        Vt[(size_t)j * n + i] = v;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) *rank = cnt;
}

}  // namespace

// CTAs for the n x n element-wise kernels behind the eigen-solver (two elements per thread at n = 128)
static unsigned small_grid(Ctx* c, int n) {
    return (unsigned)std::max<long long>(1, std::min<long long>(((long long)n * n + 511) / 512, (long long)c->sm_count * 2));
}

int eigh_jacobi(Ctx* c, const double* G, int n, double* lambda_desc, double* V, bool psd) {
    LQ_REQUIRE(c, n >= 1 && n <= 2048, LQ_ERR_UNSUPPORTED, "eigen-solver supports n <= 2048 (got %d)", n);
    const int max_sweeps = 40;
    // a pair is rotated while |a_pq| > rel_tol * sqrt(a_pp a_qq); 4 eps stops the tail of sweeps that only chase
    // rounding noise (eigenvalues move by O(a_pq^2 / gap), the eigenvector basis stays a product of exact rotations)
    const double rel_tol = 4.0 * 1.1102230246251565e-16;
    DevBuf Aw, rot, nr, lam, Vraw, ptab;
    LQ_TRY(nr.alloc(c, 16));
    LQ_TRY(lam.alloc(c, sizeof(double) * n));
    LQ_TRY(Vraw.alloc(c, sizeof(double) * (size_t)n * n));
    if (n <= 128 && !c->env_jacobi_two_sided) {
        // one-sided kernel: columns in shared memory, padded to a multiple of 16
        const int ne = (n + 15) / 16 * 16;
        LQ_TRY(Aw.alloc(c, sizeof(double) * (size_t)ne * ne));
        LQ_TRY(rot.alloc(c, sizeof(double2) * (size_t)(max_sweeps + 1) * jacobi1s_steps_per_sweep(ne) * 64));
        LQ_TRY(ptab.alloc(c, sizeof(unsigned short) * (size_t)jacobi1s_steps_per_sweep(ne) * 64));
        const int direct = psd ? 1 : 0;
        const size_t smem = sizeof(double) * (size_t)ne * ne;
        if (ne == 128)
            LQ_TRY(launch<jacobi1s_kernel<8>>(c, 1, 512, smem, c->stream, 128 * 128 * 8, G, n, ne, rot.as<double2>(), max_sweeps,
                                              rel_tol, nr.as<int>(), Aw.as<double>(), ptab.as<unsigned short>(), lam.as<double>(),
                                              direct));
        else
            LQ_TRY(launch<jacobi1s_kernel<0>>(c, 1, 512, smem, c->stream, 128 * 128 * 8, G, n, ne, rot.as<double2>(), max_sweeps,
                                              rel_tol, nr.as<int>(), Aw.as<double>(), ptab.as<unsigned short>(), lam.as<double>(),
                                              direct));
        LQ_TRY(launch<jacobi1s_apply_kernel>(c, (n + 3) / 4, 128, 0, c->stream, 0, rot.as<double2>(), nr.as<int>(),
                                             ptab.as<unsigned short>(), n, ne, Vraw.as<double>()));
        if (direct)
            LQ_TRY(launch<eigvec_from_b_kernel>(c, small_grid(c, n), 256, 0, c->stream, 0, Aw.as<double>(), ne, lam.as<double>(),
                                                nr.as<int>(), n, Vraw.as<double>()));
        LQ_TRY(launch<eig_rayleigh_kernel>(c, (n + 7) / 8, 256, 0, c->stream, 0, Aw.as<double>(), ne, Vraw.as<double>(), n,
                                           nr.as<int>(), lam.as<double>()));
        return launch<eig_sort_kernel>(c, small_grid(c, n), 256, sizeof(int) * n, c->stream, 0, lam.as<double>(), Vraw.as<double>(),
                                       n, lambda_desc, V);
    }
    const int ne = (n + 1) & ~1, ld = ne | 1, half = ne / 2;
    const size_t need = ((size_t)ne * ld + 4) * sizeof(double) + (size_t)half * sizeof(double2) + 64;
    const int use_global = need + 9216 > (size_t)c->max_smem;  // 9 KB of static shared memory in the kernel
    LQ_TRY(Aw.alloc(c, use_global ? sizeof(double) * (size_t)ne * ld : 16));
    LQ_TRY(rot.alloc(c, sizeof(double2) * (size_t)max_sweeps * (ne - 1 > 0 ? ne - 1 : 1) * (half > 0 ? half : 1)));
    const size_t smem = use_global ? (size_t)half * sizeof(double2) + 64 : need;
    LQ_TRY(launch<jacobi_kernel>(c, 1, 1024, smem, c->stream, SMEM_OPT_IN_REST, G, n, Aw.as<double>(), use_global,
                                 rot.as<double2>(), max_sweeps, rel_tol, nr.as<int>(), lam.as<double>()));
    LQ_TRY(launch<jacobi_apply_kernel>(c, n, 256, sizeof(double) * (ne + 2), c->stream, 0, rot.as<double2>(), nr.as<int>(), n, ne,
                                       Vraw.as<double>()));
    return launch<eig_sort_kernel>(c, small_grid(c, n), 256, sizeof(int) * n, c->stream, 0, lam.as<double>(), Vraw.as<double>(), n,
                                   lambda_desc, V);
}

int svd_gram_local(Ctx* c, const double* A, long long m, int n, double tol, double* U, double* s, double* Vt,
                   int* rank_host, bool sharded, int* rank_dev) {
    LQ_REQUIRE(c, m >= 1 && n >= 1, LQ_ERR_SHAPE, "svd: bad shape %lld x %d", m, n);
    LQ_REQUIRE(c, m < (1LL << 31), LQ_ERR_SHAPE, "svd: more than 2^31 rows per device not supported");
    DevBuf G, lam, V, M2, rk;
    LQ_TRY(G.alloc(c, sizeof(double) * (size_t)n * n));
    LQ_TRY(lam.alloc(c, sizeof(double) * n));
    LQ_TRY(V.alloc(c, sizeof(double) * (size_t)n * n));
    LQ_TRY(M2.alloc(c, sizeof(double) * (size_t)n * n));
    LQ_TRY(rk.alloc(c, 16));
    LQ_TRY(gram(c, A, n, m, n, G.as<double>()));                               // svd.py:42
    if (sharded) LQ_TRY(comm_allreduce_sum(c, G.as<double>(), (long long)n * n));
    LQ_TRY(eigh_jacobi(c, G.as<double>(), n, lam.as<double>(), V.as<double>(), true)); // svd.py:46-51 (G = A^T A is PSD)
    LQ_TRY(launch<svd_post_kernel>(c, small_grid(c, n), 256, sizeof(double) * n, c->stream, 0, lam.as<double>(), V.as<double>(), n,
                                   tol, s, M2.as<double>(), Vt, rk.as<int>()));
    LQ_TRY(gemm(c, false, false, m, n, n, 1.0, A, n, M2.as<double>(), n, 0.0, U, n));  // svd.py:61-64
    if (rank_dev) LQ_CUDA(c, cudaMemcpyAsync(rank_dev, rk.p, sizeof(int), cudaMemcpyDeviceToDevice, c->stream));
    if (rank_host) {
        LQ_CUDA(c, cudaMemcpyAsync(rank_host, rk.p, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
        LQ_CUDA(c, cudaStreamSynchronize(c->stream));
    }
    return LQ_OK;
}

// ------------------------------------------------------------------ counter-based standard-normal generator
// Philox4x32-10 (Salmon et al., SC'11: counter = element group, key = seed) + Box-Muller; four doubles per counter.
// The stream depends only on (seed, element index): any grid shape and any device produce the same numbers.
__device__ __forceinline__ void philox4x32_10(uint32_t (&ctr)[4], uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, ctr[0]), lo0 = 0xD2511F53u * ctr[0];
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, ctr[2]), lo1 = 0xCD9E8D57u * ctr[2];
        const uint32_t n0 = hi1 ^ ctr[1] ^ k0, n2 = hi0 ^ ctr[3] ^ k1;
        ctr[0] = n0;
        ctr[1] = lo1;
        ctr[2] = n2;
        ctr[3] = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
}
__global__ void __launch_bounds__(256) philox_normal_kernel(double* __restrict__ out, long long count, unsigned long long seed) {
    const long long groups = (count + 3) / 4;
    for (long long gidx = (long long)blockIdx.x * blockDim.x + threadIdx.x; gidx < groups; gidx += (long long)gridDim.x * blockDim.x) {
        double z[4];
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            uint32_t ctr[4] = {(uint32_t)gidx, (uint32_t)((unsigned long long)gidx >> 32), (uint32_t)half, 0x6c696e61u};
            philox4x32_10(ctr, (uint32_t)seed, (uint32_t)(seed >> 32));
            // two uniforms in (0, 1] / [0, 1) with 53 / 32 bits, one Box-Muller pair
            const unsigned long long b = ((unsigned long long)ctr[0] << 32) | ctr[1];
            const double u1 = ((double)(b >> 11) + 1.0) * (1.0 / 9007199254740992.0);
            const double u2 = ((double)ctr[2] * 4294967296.0 + (double)ctr[3]) * (1.0 / 18446744073709551616.0);
            const double rad = sqrt(-2.0 * log(u1));
            double sn, cs;
            sincospi(2.0 * u2, &sn, &cs);
            z[2 * half] = rad * cs;
            z[2 * half + 1] = rad * sn;
        }
#pragma unroll
        for (int e = 0; e < 4; ++e)
            if (4 * gidx + e < count) out[4 * gidx + e] = z[e];
    }
}

}  // namespace lq

using namespace lq;

extern "C" {

int lq_gram_dev(lq_ctx* h, const double* A, int64_t m, int n, double* G) {
    Ctx* c = as_ctx(h);
    if (!c) return LQ_ERR_ARG;
    LQ_REQUIRE(c, m >= 1 && n >= 1 && m < (1LL << 31), LQ_ERR_SHAPE, "gram: bad shape");
    LQ_CUDA(c, cudaSetDevice(c->device));
    return gram(c, A, n, m, n, G);
}
int lq_eigh_dev(lq_ctx* h, const double* G, int n, double* lambda_desc, double* V) {
    Ctx* c = as_ctx(h);
    if (!c) return LQ_ERR_ARG;
    LQ_REQUIRE(c, n >= 1 && n <= 2048, LQ_ERR_SHAPE, "eigh: n must be in [1, 2048] (got %d)", n);
    LQ_CUDA(c, cudaSetDevice(c->device));
    return eigh_jacobi(c, G, n, lambda_desc, V);
}
int lq_svd_gram_dev(lq_ctx* h, const double* A, int64_t m, int n, double tol, double* U, double* s, double* Vt,
                    int* rank_host) {
    Ctx* c = as_ctx(h);
    if (!c) return LQ_ERR_ARG;
    LQ_REQUIRE(c, m >= n, LQ_ERR_SHAPE, "svd_gram needs m >= n (transpose on the host side, svd.py:37-39)");
    LQ_CUDA(c, cudaSetDevice(c->device));
    return svd_gram_local(c, A, m, n, tol, U, s, Vt, rank_host, false);
}
int lq_svd_gram_sharded_dev(lq_ctx* h, const double* A, int64_t m, int n, double tol, double* U, double* s, double* Vt,
                            int* rank_host) {
    Ctx* c = as_ctx(h);
    if (!c) return LQ_ERR_ARG;
    LQ_CUDA(c, cudaSetDevice(c->device));
    return svd_gram_local(c, A, m, n, tol, U, s, Vt, rank_host, true);
}
// linalg/svd.py:67-76 on the device: orthonormal completion of U (host, m x n, first `rank` columns
// valid) from the candidate directions Z: drawn by the caller (host, m x (n - rank): upstream draws them from the global
// np.random) or, with a seed, generated on the device (no upload; deterministic -- SURVEY.md section 8f-1).
static int svd_complete_impl(lq_ctx* h, double* U, int64_t m, int n, int rank, const double* Z, bool seeded, unsigned long long seed) {
    Ctx* c = as_ctx(h);
    if (!c) return LQ_ERR_ARG;
    const int k = n - rank;
    LQ_REQUIRE(c, m >= n && rank >= 0 && k >= 1 && U && (Z || seeded), LQ_ERR_SHAPE, "svd_complete: bad arguments");
    LQ_REQUIRE(c, m < (1LL << 31), LQ_ERR_SHAPE, "svd_complete: too many rows");
    LQ_CUDA(c, cudaSetDevice(c->device));
    DevBuf dU, dZ, dQ, dR, dW;
    LQ_TRY(dU.alloc(c, sizeof(double) * (size_t)m * n));
    LQ_TRY(dZ.alloc(c, sizeof(double) * (size_t)m * k));
    LQ_TRY(dQ.alloc(c, sizeof(double) * (size_t)m * k));
    LQ_TRY(dR.alloc(c, sizeof(double) * (size_t)k * k));
    LQ_TRY(dW.alloc(c, sizeof(double) * (size_t)n * k));
    LQ_CUDA(c, cudaMemcpyAsync(dU.p, U, sizeof(double) * (size_t)m * n, cudaMemcpyHostToDevice, c->stream));
    if (seeded) {
        const long long count = (long long)m * k;
        LQ_TRY(launch<philox_normal_kernel>(c, grid_for(c, (count + 3) / 4), 256, 0, c->stream, 0, dZ.as<double>(), count, seed));
    } else {
        LQ_CUDA(c, cudaMemcpyAsync(dZ.p, Z, sizeof(double) * (size_t)m * k, cudaMemcpyHostToDevice, c->stream));
    }
    LQ_TRY(lq_householder_qr_dev(h, dZ.as<double>(), (int)m, k, dQ.as<double>(), dR.as<double>()));          // svd.py:69
    if (rank > 0) {
        // Q -= U_r (U_r^T Q)                                                                                // svd.py:71-72
        LQ_TRY(gemm(c, true, false, rank, k, (int)m, 1.0, dU.as<double>(), n, dQ.as<double>(), k, 0.0, dW.as<double>(), k));
        LQ_TRY(gemm(c, false, false, m, k, rank, -1.0, dU.as<double>(), n, dW.as<double>(), k, 1.0, dQ.as<double>(), k));
    }
    LQ_TRY(lq_householder_qr_dev(h, dQ.as<double>(), (int)m, k, dZ.as<double>(), dR.as<double>()));          // svd.py:74
    // U[:, rank:] = Z
    LQ_CUDA(c, cudaMemcpy2DAsync(U + rank, sizeof(double) * n, dZ.p, sizeof(double) * k, sizeof(double) * k, (size_t)m,
                                 cudaMemcpyDeviceToHost, c->stream));
    LQ_CUDA(c, cudaStreamSynchronize(c->stream));
    return LQ_OK;
}
int lq_svd_complete(lq_ctx* h, double* U, int64_t m, int n, int rank, const double* Z) {
    return svd_complete_impl(h, U, m, n, rank, Z, false, 0ULL);
}
int lq_svd_complete_seeded(lq_ctx* h, double* U, int64_t m, int n, int rank, uint64_t seed) {
    return svd_complete_impl(h, U, m, n, rank, nullptr, true, (unsigned long long)seed);
}
int lq_random_normal_dev(lq_ctx* h, double* out, int64_t count, uint64_t seed) {
    Ctx* c = as_ctx(h);
    if (!c) return LQ_ERR_ARG;
    LQ_REQUIRE(c, count >= 0 && (count == 0 || out), LQ_ERR_ARG, "random_normal: bad arguments");
    if (count == 0) return LQ_OK;
    LQ_CUDA(c, cudaSetDevice(c->device));
    return launch<philox_normal_kernel>(c, grid_for(c, (count + 3) / 4), 256, 0, c->stream, 0, out, count,
                                        (unsigned long long)seed);
}

}  // extern "C"

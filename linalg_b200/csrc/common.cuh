// Shared device/host helpers for the linalg_b200 kernels (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>

namespace lq {

constexpr double kEps = 1e-12;  // reference linalg/utils.py:9 (absolute threshold)

// ------------------------------------------------------------------ errors
// 0 ok; <0 argument/shape error (-> ValueError); >0 CUDA/NCCL status (-> RuntimeError)
enum : int {
    LQ_OK = 0,
    LQ_ERR_ARG = -1,
    LQ_ERR_SHAPE = -2,
    LQ_ERR_UNSUPPORTED = -3,
    LQ_ERR_NOMEM = -4,
    LQ_ERR_NCCL_MISSING = -5,
    LQ_ERR_CUDA_BASE = 1000,   // 1000 + cudaError_t
    LQ_ERR_NCCL_BASE = 5000,   // 5000 + ncclResult_t
};

struct Ctx;
void set_error(Ctx* c, const char* fmt, ...);

#define LQ_CUDA(ctx, expr)                                                                  \
    do {                                                                                    \
        cudaError_t _e = (expr);                                                            \
        if (_e != cudaSuccess) {                                                            \
            ::lq::set_error((ctx), "%s:%d: %s -> %s", __FILE__, __LINE__, #expr,            \
                            cudaGetErrorString(_e));                                        \
            return ::lq::LQ_ERR_CUDA_BASE + (int)_e;                                        \
        }                                                                                   \
    } while (0)

#define LQ_CHECK_LAUNCH(ctx) LQ_CUDA(ctx, cudaGetLastError())

#define LQ_REQUIRE(ctx, cond, code, ...)                                                    \
    do {                                                                                    \
        if (!(cond)) {                                                                      \
            ::lq::set_error((ctx), __VA_ARGS__);                                            \
            return (code);                                                                  \
        }                                                                                   \
    } while (0)

#define LQ_TRY(expr)                                                                        \
    do {                                                                                    \
        int _rc = (expr);                                                                   \
        if (_rc != 0) return _rc;                                                           \
    } while (0)

// Diagnostic environment switches are read ONCE per call site (never on a hot path: a blocked QR issues thousands of GEMMs)
#define LQ_ENV_ONCE(name) ([]() -> bool { static const bool v = ::getenv(name) != nullptr; return v; }())

// ------------------------------------------------------------------ device math helpers
__device__ __forceinline__ double rcp_seed(double x) {
    double y;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    return y;
}
__device__ __forceinline__ double rsqrt_seed(double x) {
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    return y;
}
// 1/x for normal, finite, non-zero x: MUFU seed + IT Newton steps (branch free).
template <int IT>
__device__ __forceinline__ double rcp_nr_t(double x) {
    double y = rcp_seed(x);
#pragma unroll
    for (int it = 0; it < IT; ++it) {
        const double e = fma(-x, y, 1.0);
        y = fma(y, e, y);
    }
    return y;
}
// 1/sqrt(x) for normal positive x.
template <int IT>
__device__ __forceinline__ double rsqrt_nr_t(double x) {
    double y = rsqrt_seed(x);
    const double hx = 0.5 * x;
#pragma unroll
    for (int it = 0; it < IT; ++it) {
        const double e = fma(-hx * y, y, 0.5);  // 0.5 - 0.5*x*y^2
        y = fma(y, e, y);
    }
    return y;
}
// sqrt(x) (x > 0, normal) from rsqrt with one correction step; also returns 1/sqrt(x).
template <int IT>
__device__ __forceinline__ double sqrt_nr_t(double x, double& rinv) {
    rinv = rsqrt_nr_t<IT>(x);
    const double s = x * rinv;
    const double res = fma(-s, s, x);
    return fma(res, 0.5 * rinv, s);
}
__device__ __forceinline__ double rcp_nr(double x) { return rcp_nr_t<3>(x); }
__device__ __forceinline__ double rsqrt_nr(double x) { return rsqrt_nr_t<3>(x); }
__device__ __forceinline__ double sqrt_nr(double x, double& rinv) { return sqrt_nr_t<3>(x, rinv); }

__device__ __forceinline__ double ld_stream(const double* p) {
    double v;
    asm volatile("ld.global.nc.L1::no_allocate.f64 %0, [%1];" : "=d"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ void st_stream(double* p, double v) {
    asm volatile("st.global.L1::no_allocate.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory");
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// FP64 tensor-core MMA (legacy warp-level path; tcgen05 has no f64 kind on sm_100a).
// D(16x8) += A(16x8) * B(8x8).  Fragment layout (lane l, g = l/4, t = l%4):
//   a0=A[g][t] a1=A[g+8][t] a2=A[g][t+4] a3=A[g+8][t+4];  b0=B[t][g] b1=B[t+4][g]
//   c0=C[g][2t] c1=C[g][2t+1] c2=C[g+8][2t] c3=C[g+8][2t+1]
__device__ __forceinline__ void dmma_16x8x8(double (&c)[4], const double (&a)[4], const double (&b)[2]) {
    asm volatile(
        "mma.sync.aligned.m16n8k8.row.col.f64.f64.f64.f64 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, "
        "{%0,%1,%2,%3};\n"
        : "+d"(c[0]), "+d"(c[1]), "+d"(c[2]), "+d"(c[3])
        : "d"(a[0]), "d"(a[1]), "d"(a[2]), "d"(a[3]), "d"(b[0]), "d"(b[1]));
}
// D(8x8) += A(8x4) * B(4x8):  a=A[g][t], b=B[t][g], c0=C[g][2t], c1=C[g][2t+1]
__device__ __forceinline__ void dmma_8x8x4(double (&c)[2], double a, double b) {
    asm volatile(
        "mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
        : "+d"(c[0]), "+d"(c[1])
        : "d"(a), "d"(b));
}

// ------------------------------------------------------------------ mbarrier / bulk-copy (TMA engine) helpers
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {
    }
}
// 1-D bulk async copy global -> shared (TMA engine, SASS UBLKCP); bytes % 16 == 0, both 16B aligned.
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(smem_dst)),
        "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}
// 1-D bulk async copy shared -> global.
__device__ __forceinline__ void bulk_s2g(void* gmem_dst, const void* smem_src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gmem_dst),
                 "r"(smem_u32(smem_src)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void bulk_wait() {
    asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ------------------------------------------------------------------ cluster helpers
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ uint32_t cluster_nctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_arrive() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
}
__device__ __forceinline__ void cluster_wait() {
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
    cluster_arrive();
    cluster_wait();
}
// map a local shared address to the same offset in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_shared(uint32_t local_addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void st_cluster_f64(uint32_t addr, double v) {
    asm volatile("st.shared::cluster.f64 [%0], %1;" ::"r"(addr), "d"(v) : "memory");
}
__device__ __forceinline__ double ld_cluster_f64(uint32_t addr) {
    double v;
    asm volatile("ld.shared::cluster.f64 %0, [%1];" : "=d"(v) : "r"(addr) : "memory");
    return v;
}

// ------------------------------------------------------------------ Jacobi round-robin ("circle") ordering
// Pair k (0 <= k < n_even / 2) of round `round` (0 <= round < n_even - 1): every index meets every other once per sweep.
__device__ __forceinline__ void rr_pair(int n_even, int round, int k, int& p, int& q) {
    // players 0..n_even-2 on a circle, player n_even-1 fixed
    const int mod = n_even - 1;
    int a, b;
    if (k == 0) {
        a = n_even - 1;
        b = round % mod;
    } else {
        a = (round + k) % mod;
        b = (round - k + mod) % mod;
    }
    p = min(a, b);
    q = max(a, b);
}

// ------------------------------------------------------------------ descending eigenvalue order
// Whether eigenvalue a (index ia) comes before b (index ib): NaN first (where the reference's np.argsort(lam)[::-1] puts it),
// then descending, equal values by index.  A strict total order even with NaN, so ranking by counting is a permutation; a
// bare (b > a) || (b == a && ib < ia) is false both ways for NaN and gives several eigenvalues the same rank.
__device__ __forceinline__ bool eig_desc_before(double a, int ia, double b, int ib) {
    const bool na = isnan(a), nb = isnan(b);
    if (na != nb) return na;
    return (!na && a > b) || ((na || a == b) && ia < ib);
}

// s = sqrt(max(lambda, 0)) that keeps a NaN eigenvalue NaN, as the reference's np.sqrt(np.clip(lam, 0, None)) does (fmax
// alone drops the NaN operand and would report sigma = 0 for a non-finite matrix)
__device__ __forceinline__ double sqrt_clip0(double lam) { return sqrt(isnan(lam) ? lam : fmax(lam, 0.0)); }

// the eigenvalue of a matrix with a NaN or infinite entry (the default quiet NaN, one payload on every route)
__device__ __forceinline__ double eig_nan() { return __longlong_as_double(0x7ff8000000000000LL); }

}  // namespace lq

// Context lifecycle, memory, timing and roofline probes of the linalg_b200 C ABI.
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <mutex>

#include "../../include/linalg_b200.h"
#include "ops.cuh"

namespace lq {

std::string& global_error() {
    static thread_local std::string e;
    return e;
}

void set_error(Ctx* c, const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (c) c->err = buf;
    global_error() = buf;
}

// ------------------------------------------------------------------ probe kernels
// FP64 FMA peak: 8 independent chains per thread, fully unrolled.
__global__ void __launch_bounds__(256) probe_dfma_kernel(double* out, int iters, double seed) {
    double a[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) a[k] = seed + k + threadIdx.x * 1e-9;
    const double m = 1.0000001, c = 1e-9;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int u = 0; u < 8; ++u)
#pragma unroll
            for (int k = 0; k < 8; ++k) a[k] = fma(a[k], m, c);
    }
    double s = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) s += a[k];
    if (s == 123.456) out[0] = s;
}
// FP64 tensor peak: m16n8k8 DMMA, 8 independent accumulator tiles per warp.
__global__ void __launch_bounds__(256) probe_dmma_kernel(double* out, int iters, double seed) {
    double c[8][4];
#pragma unroll
    for (int k = 0; k < 8; ++k)
#pragma unroll
        for (int e = 0; e < 4; ++e) c[k][e] = seed + e;
    double a[4] = {1.0 + seed, 0.5, 0.25, 0.125};
    double b[2] = {1e-9, 2e-9};
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
            for (int k = 0; k < 8; ++k) dmma_16x8x8(c[k], a, b);
    }
    double s = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k)
#pragma unroll
        for (int e = 0; e < 4; ++e) s += c[k][e];
    if (s == 123.456) out[0] = s;
}
// both pipes at once: does DMMA run beside DFMA or on the same datapath?
__global__ void __launch_bounds__(256) probe_mixed_kernel(double* out, int iters, double seed) {
    double c[4][4];
    double a8[8];
#pragma unroll
    for (int k = 0; k < 4; ++k)
#pragma unroll
        for (int e = 0; e < 4; ++e) c[k][e] = seed + e;
#pragma unroll
    for (int k = 0; k < 8; ++k) a8[k] = seed + k;
    double a[4] = {1.0 + seed, 0.5, 0.25, 0.125};
    double b[2] = {1e-9, 2e-9};
    const double m = 1.0000001, cc = 1e-9;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int u = 0; u < 4; ++u) {
#pragma unroll
            for (int k = 0; k < 4; ++k) dmma_16x8x8(c[k], a, b);
#pragma unroll
            for (int r = 0; r < 4; ++r)
#pragma unroll
                for (int k = 0; k < 8; ++k) a8[k] = fma(a8[k], m, cc);
        }
    }
    double s = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k)
#pragma unroll
        for (int e = 0; e < 4; ++e) s += c[k][e];
#pragma unroll
    for (int k = 0; k < 8; ++k) s += a8[k];
    if (s == 123.456) out[0] = s;
}
__global__ void __launch_bounds__(256) probe_copy_kernel(const double4* __restrict__ src, double4* __restrict__ dst,
                                                         size_t n4) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (; i < n4; i += stride) dst[i] = src[i];
}
// latency of a dependent DFMA chain (cycles per DFMA), one warp
__global__ void probe_dfma_latency_kernel(double* out, double seed) {
    double a = seed;
    const double m = 1.0000001, c = 1e-9;
    long long t0 = clock64();
#pragma unroll 1
    for (int it = 0; it < 64; ++it) {
#pragma unroll
        for (int u = 0; u < 64; ++u) a = fma(a, m, c);
    }
    long long t1 = clock64();
    if (threadIdx.x == 0) {
        out[0] = (double)(t1 - t0) / (64.0 * 64.0);
        out[1] = a;
    }
}
// accuracy of the MUFU seeds and of the Newton-refined reciprocal / rsqrt / sqrt used by the kernels
__global__ void probe_seed_accuracy_kernel(double* out) {
    double e_rcp = 0, e_rsq = 0, e_rcp_nr = 0, e_rsq_nr = 0, e_sqrt_nr = 0, e_rcp2 = 0, e_rsq2 = 0;
    unsigned long long st = 0x9E3779B97F4A7C15ull * (threadIdx.x + 1 + 1024ull * blockIdx.x);
    for (int it = 0; it < 4096; ++it) {
        st = st * 6364136223846793005ull + 1442695040888963407ull;
        const double u = (double)(st >> 11) * (1.0 / 9007199254740992.0);
        const int ex = (int)((st >> 3) % 40) - 20;
        const double x = ldexp(0.5 + u, ex * 3);
        const double r_true = 1.0 / x, q_true = 1.0 / sqrt(x);
        e_rcp = fmax(e_rcp, fabs(rcp_seed(x) - r_true) / r_true);
        e_rsq = fmax(e_rsq, fabs(rsqrt_seed(x) - q_true) / q_true);
        e_rcp_nr = fmax(e_rcp_nr, fabs(rcp_nr(x) - r_true) / r_true);
        e_rsq_nr = fmax(e_rsq_nr, fabs(rsqrt_nr(x) - q_true) / q_true);
        double ri;
        e_sqrt_nr = fmax(e_sqrt_nr, fabs(sqrt_nr(x, ri) - sqrt(x)) / sqrt(x));
        {   // two Newton steps only
            double y = rcp_seed(x);
            double e = fma(-x, y, 1.0); y = fma(y, e, y);
            e = fma(-x, y, 1.0); y = fma(y, e, y);
            e_rcp2 = fmax(e_rcp2, fabs(y - r_true) / r_true);
            double z = rsqrt_seed(x); const double hx = 0.5 * x;
            double f = fma(-hx * z, z, 0.5); z = fma(z, f, z);
            f = fma(-hx * z, z, 0.5); z = fma(z, f, z);
            e_rsq2 = fmax(e_rsq2, fabs(z - q_true) / q_true);
        }
    }
    double v[7] = {e_rcp, e_rsq, e_rcp_nr, e_rsq_nr, e_sqrt_nr, e_rcp2, e_rsq2};
    for (int k = 0; k < 7; ++k) {
        double m = v[k];
        for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
        if ((threadIdx.x & 31) == 0) atomicMax((unsigned long long*)&out[k], (unsigned long long)__double_as_longlong(m));
    }
}
__global__ void fill_kernel(double* p, size_t n, double v) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) p[i] = v;
}

}  // namespace lq

using namespace lq;

extern "C" {

const char* lq_version(void) { return "linalg_b200 0.1.0 (sm_100a)"; }

int lq_device_count(int* count) {
    if (!count) return LQ_ERR_ARG;
    cudaError_t e = cudaGetDeviceCount(count);
    if (e != cudaSuccess) {
        *count = 0;
        set_error(nullptr, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
        return LQ_ERR_CUDA_BASE + (int)e;
    }
    return LQ_OK;
}

int lq_create(int device, lq_ctx** out) {
    if (!out) return LQ_ERR_ARG;
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        set_error(nullptr, "no CUDA device available (%s); linalg_b200 has no CPU fallback",
                  e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
        return LQ_ERR_CUDA_BASE + (int)(e != cudaSuccess ? e : cudaErrorNoDevice);
    }
    if (device < 0 || device >= n) {
        set_error(nullptr, "device %d out of range [0, %d)", device, n);
        return LQ_ERR_ARG;
    }
    // owns the context until every resource exists: a failing CUDA call below returns through lq_destroy
    struct Guard {
        Ctx* c;
        ~Guard() {
            if (c) {
                std::string keep = c->err;
                lq_destroy(c);
                if (!keep.empty()) global_error() = keep;
            }
        }
    } guard{new Ctx()};
    Ctx* c = guard.c;
    c->device = device;
    LQ_CUDA(c, cudaSetDevice(device));
    LQ_CUDA(c, cudaGetDeviceProperties(&c->prop, device));
    if (c->prop.major < 10) {
        set_error(nullptr, "device %d is sm_%d%d; linalg_b200 is built for sm_100a only", device, c->prop.major,
                  c->prop.minor);
        return LQ_ERR_UNSUPPORTED;
    }
    c->sm_count = c->prop.multiProcessorCount;
    c->max_smem = (int)c->prop.sharedMemPerBlockOptin;
    LQ_TRY(measure_max_cluster(c));
    // the context stream carries the latency-bound chains (panel factorisations); the side lanes carry bulk
    // work that overlaps with them, so the main stream gets the higher scheduling priority
    int prio_lo = 0, prio_hi = 0;
    LQ_CUDA(c, cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
    LQ_CUDA(c, cudaStreamCreateWithPriority(&c->stream, cudaStreamNonBlocking, prio_hi));
    LQ_CUDA(c, cudaStreamCreateWithFlags(&c->lane[0], cudaStreamNonBlocking));
    for (int i = 1; i < 3; ++i) LQ_CUDA(c, cudaStreamCreateWithPriority(&c->lane[i], cudaStreamNonBlocking, prio_hi));
    LQ_CUDA(c, cudaStreamCreateWithFlags(&c->lane[3], cudaStreamNonBlocking));
    for (int i = 0; i < 16; ++i) LQ_CUDA(c, cudaEventCreate(&c->ev[i]));
    // keep freed scratch cached in the stream-ordered pool
    cudaMemPool_t pool;
    LQ_CUDA(c, cudaDeviceGetDefaultMemPool(&pool, device));
    unsigned long long thr = ~0ull;
    LQ_CUDA(c, cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr));
    c->env_tsqr_householder = getenv("LINALG_B200_TSQR_HOUSEHOLDER") != nullptr;
    c->env_jacobi_two_sided = getenv("LINALG_B200_JACOBI_TWO_SIDED") != nullptr;
    c->env_no_graph = getenv("LINALG_B200_NO_GRAPH") != nullptr;
    guard.c = nullptr;
    *out = c;
    return LQ_OK;
}

int lq_destroy(lq_ctx* h) {
    Ctx* c = as_ctx(h);
    if (!c) return LQ_OK;
    cudaSetDevice(c->device);
    lq_comm_destroy(h);
    cudaStreamSynchronize(c->stream);
    for (auto& g : c->graphs)
        if (g.exec) cudaGraphExecDestroy(g.exec);
    c->graphs.clear();
    if (c->flush_buf) cudaFree(c->flush_buf);
    for (int i = 0; i < 16; ++i)
        if (c->ev[i]) cudaEventDestroy(c->ev[i]);
    for (int i = 0; i < 4; ++i)
        if (c->lane[i]) cudaStreamDestroy(c->lane[i]);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
    return LQ_OK;
}

int lq_set_option(lq_ctx* h, const char* name, int value) {
    Ctx* c = as_ctx(h);
    if (!c || !name) return LQ_ERR_ARG;
    const std::string n(name);
    if (n == "TSQR_HOUSEHOLDER") c->env_tsqr_householder = value != 0;
    else if (n == "JACOBI_TWO_SIDED") c->env_jacobi_two_sided = value != 0;
    else {
        set_error(c, "lq_set_option: unknown option '%s'", name);
        return LQ_ERR_ARG;
    }
    return LQ_OK;
}

const char* lq_last_error(lq_ctx* h) {
    Ctx* c = as_ctx(h);
    return c ? c->err.c_str() : global_error().c_str();
}

int lq_device_props(lq_ctx* h, int64_t props[8]) {
    Ctx* c = as_ctx(h);
    if (!c || !props) return LQ_ERR_ARG;
    props[0] = c->sm_count;
    props[1] = c->prop.major;
    props[2] = c->prop.minor;
    props[3] = c->max_smem;
    int khz = 0;
    cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, c->device);
    props[4] = khz;
    props[5] = (int64_t)(c->prop.totalGlobalMem >> 20);
    props[6] = c->prop.l2CacheSize;
    props[7] = c->max_cluster;
    return LQ_OK;
}

int lq_malloc(lq_ctx* h, size_t bytes, void** dptr) {
    Ctx* c = as_ctx(h);
    if (!c || !dptr) return LQ_ERR_ARG;
    LQ_CUDA(c, cudaSetDevice(c->device));
    LQ_CUDA(c, cudaMalloc(dptr, bytes ? bytes : 16));
    return LQ_OK;
}
int lq_free(lq_ctx* h, void* dptr) {
    Ctx* c = as_ctx(h);
    if (!c) return LQ_ERR_ARG;
    if (dptr) LQ_CUDA(c, cudaFree(dptr));
    return LQ_OK;
}
int lq_host_alloc(size_t bytes, void** hptr) {
    if (!hptr) return LQ_ERR_ARG;
    cudaError_t e = cudaHostAlloc(hptr, bytes ? bytes : 16, cudaHostAllocPortable);
    if (e != cudaSuccess) {
        set_error(nullptr, "cudaHostAlloc(%zu): %s", bytes, cudaGetErrorString(e));
        return LQ_ERR_CUDA_BASE + (int)e;
    }
    return LQ_OK;
}
int lq_host_free(void* hptr) {
    if (hptr) cudaFreeHost(hptr);
    return LQ_OK;
}
int lq_memcpy_h2d(lq_ctx* h, void* dst, const void* src, size_t bytes) {
    Ctx* c = as_ctx(h);
    if (!c) return LQ_ERR_ARG;
    LQ_CUDA(c, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, c->stream));
    return LQ_OK;
}
int lq_memcpy_d2h(lq_ctx* h, void* dst, const void* src, size_t bytes) {
    Ctx* c = as_ctx(h);
    if (!c) return LQ_ERR_ARG;
    LQ_CUDA(c, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, c->stream));
    return LQ_OK;
}
int lq_memcpy_d2d(lq_ctx* h, void* dst, const void* src, size_t bytes) {
    Ctx* c = as_ctx(h);
    if (!c) return LQ_ERR_ARG;
    LQ_CUDA(c, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, c->stream));
    return LQ_OK;
}
int lq_memset(lq_ctx* h, void* dst, int value, size_t bytes) {
    Ctx* c = as_ctx(h);
    if (!c) return LQ_ERR_ARG;
    LQ_CUDA(c, cudaMemsetAsync(dst, value, bytes, c->stream));
    return LQ_OK;
}
int lq_sync(lq_ctx* h) {
    Ctx* c = as_ctx(h);
    if (!c) return LQ_ERR_ARG;
    LQ_CUDA(c, cudaStreamSynchronize(c->stream));
    return LQ_OK;
}
int lq_event_record(lq_ctx* h, int slot) {
    Ctx* c = as_ctx(h);
    if (!c || slot < 0 || slot >= 16) return LQ_ERR_ARG;
    LQ_CUDA(c, cudaEventRecord(c->ev[slot], c->stream));
    return LQ_OK;
}
int lq_event_elapsed_ms(lq_ctx* h, int a, int b, float* ms) {
    Ctx* c = as_ctx(h);
    if (!c || !ms || a < 0 || a >= 16 || b < 0 || b >= 16) return LQ_ERR_ARG;
    LQ_CUDA(c, cudaEventSynchronize(c->ev[b]));
    LQ_CUDA(c, cudaEventElapsedTime(ms, c->ev[a], c->ev[b]));
    return LQ_OK;
}
int lq_flush_l2(lq_ctx* h) {
    Ctx* c = as_ctx(h);
    if (!c) return LQ_ERR_ARG;
    LQ_CUDA(c, cudaSetDevice(c->device));
    const size_t bytes = (size_t)256 << 20;
    if (!c->flush_buf) LQ_CUDA(c, cudaMalloc(&c->flush_buf, bytes));
    fill_kernel<<<c->sm_count * 8, 256, 0, c->stream>>>((double*)c->flush_buf, bytes / 8, 1.0);
    LQ_CHECK_LAUNCH(c);
    return LQ_OK;
}
int64_t lq_kernel_launches(lq_ctx* h) {
    Ctx* c = as_ctx(h);
    return c ? c->launches : 0;
}

int lq_probe(lq_ctx* h, int kind, double* result) {
    Ctx* c = as_ctx(h);
    if (!c || !result) return LQ_ERR_ARG;
    LQ_CUDA(c, cudaSetDevice(c->device));
    cudaEvent_t e0 = c->ev[14], e1 = c->ev[15];
    float ms = 0, best = 1e30f;
    if (kind == 0 || kind == 1 || kind == 3) {
        DevBuf out;
        LQ_TRY(out.alloc(c, 64));
        const int iters = 4096, blocks = c->sm_count * 8, threads = 256;
        for (int rep = 0; rep < 6; ++rep) {
            LQ_CUDA(c, cudaEventRecord(e0, c->stream));
            if (kind == 0) probe_dfma_kernel<<<blocks, threads, 0, c->stream>>>(out.as<double>(), iters, 1.0);
            else if (kind == 1) probe_dmma_kernel<<<blocks, threads, 0, c->stream>>>(out.as<double>(), iters, 1.0);
            else probe_mixed_kernel<<<blocks, threads, 0, c->stream>>>(out.as<double>(), iters, 1.0);
            LQ_CHECK_LAUNCH(c);
            LQ_CUDA(c, cudaEventRecord(e1, c->stream));
            LQ_CUDA(c, cudaEventSynchronize(e1));
            LQ_CUDA(c, cudaEventElapsedTime(&ms, e0, e1));
            if (rep > 0 && ms < best) best = ms;
        }
        double flops;
        if (kind == 0) flops = 2.0 * 64 * iters * (double)blocks * threads;
        else if (kind == 1) flops = 2.0 * (16 * 8 * 8) * 32.0 * iters * (double)blocks * (threads / 32);
        else
            flops = (2.0 * (16 * 8 * 8) * 16.0 * iters) * (double)blocks * (threads / 32) +
                    2.0 * 128 * iters * (double)blocks * threads;
        *result = flops / (best * 1e-3) / 1e12;
        return LQ_OK;
    }
    if (kind == 2) {
        const size_t bytes = (size_t)1 << 30;
        DevBuf a, b;
        LQ_TRY(a.alloc(c, bytes));
        LQ_TRY(b.alloc(c, bytes));
        fill_kernel<<<c->sm_count * 8, 256, 0, c->stream>>>(a.as<double>(), bytes / 8, 1.5);
        LQ_CHECK_LAUNCH(c);
        for (int rep = 0; rep < 6; ++rep) {
            LQ_CUDA(c, cudaEventRecord(e0, c->stream));
            probe_copy_kernel<<<c->sm_count * 16, 256, 0, c->stream>>>(a.as<double4>(), b.as<double4>(), bytes / 32);
            LQ_CHECK_LAUNCH(c);
            LQ_CUDA(c, cudaEventRecord(e1, c->stream));
            LQ_CUDA(c, cudaEventSynchronize(e1));
            LQ_CUDA(c, cudaEventElapsedTime(&ms, e0, e1));
            if (rep > 0 && ms < best) best = ms;
        }
        *result = 2.0 * bytes / (best * 1e-3) / 1e9;
        return LQ_OK;
    }
    if (kind == 4) {  // DFMA dependent-issue latency in cycles
        DevBuf out;
        LQ_TRY(out.alloc(c, 64));
        probe_dfma_latency_kernel<<<1, 32, 0, c->stream>>>(out.as<double>(), 1.0);
        LQ_CHECK_LAUNCH(c);
        double hres[2];
        LQ_CUDA(c, cudaMemcpyAsync(hres, out.p, 16, cudaMemcpyDeviceToHost, c->stream));
        LQ_CUDA(c, cudaStreamSynchronize(c->stream));
        *result = hres[0];
        return LQ_OK;
    }
    if (kind >= 10 && kind < 17) {  // seed / Newton accuracy (max relative error), see probe_seed_accuracy_kernel
        DevBuf out;
        LQ_TRY(out.alloc(c, 64));
        LQ_CUDA(c, cudaMemsetAsync(out.p, 0, 64, c->stream));
        probe_seed_accuracy_kernel<<<8, 128, 0, c->stream>>>(out.as<double>());
        LQ_CHECK_LAUNCH(c);
        double hres[8];
        LQ_CUDA(c, cudaMemcpyAsync(hres, out.p, 56, cudaMemcpyDeviceToHost, c->stream));
        LQ_CUDA(c, cudaStreamSynchronize(c->stream));
        *result = hres[kind - 10];
        return LQ_OK;
    }
    set_error(c, "lq_probe: unknown kind %d", kind);
    return LQ_ERR_ARG;
}

}  // extern "C"

// Context object behind the opaque lq_ctx handle.
#pragma once

#include <cuda_runtime.h>

#include <cstdarg>
#include <string>
#include <vector>

#include "common.cuh"

struct lq_ctx {};  // opaque tag for the C ABI

namespace lq {

struct Ctx : lq_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    // lane 0 / 1: copy-compute lanes of the host-pointer pipelines and side / aux streams of the blocked QR's look-ahead;
    // lane 2: T-merge stream of the blocked QR (lanes 1 and 2 carry latency-critical work: high priority);
    // lane 3: second trailing-update stream of the blocked QR.
    cudaStream_t lane[4] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t ev[16] = {};
    cudaDeviceProp prop{};
    int sm_count = 0;
    int max_smem = 0;        // opt-in dynamic shared memory per block
    int max_cluster = 1;     // largest cluster size the panel kernel may use (measure_max_cluster)
    std::string err;
    void* flush_buf = nullptr;
    long long launches = 0;
    // NCCL (loaded lazily with dlopen)
    void* nccl_comm = nullptr;
    int nranks = 1, rank = 0;
    // diagnostic kernel-selection switches: initialised from LINALG_B200_<NAME> when the context is created, changed with
    // lq_set_option (never read from the environment on a hot entry point)
    bool env_tsqr_householder = false, env_jacobi_two_sided = false;
    // CUDA-graph replay of the blocked QR schedule for small single matrices (launch-latency bound: 52 launches over five
    // streams at 256^2).  Keyed by shape and the caller's device pointers; state 0 = seen once (warm-up call, runs the
    // plain path so that every per-kernel attribute latch is set outside a capture), 1 = graph ready, -1 = not capturable.
    struct GraphEntry {
        int m = 0, n = 0;
        const void* A = nullptr;
        void* Q = nullptr;
        void* R = nullptr;
        cudaGraphExec_t exec = nullptr;
        long long launches = 0;
        int state = 0;
        unsigned long long stamp = 0;
    };
    std::vector<GraphEntry> graphs;
    unsigned long long graph_clock = 0;
    bool env_no_graph = false;
};

std::string& global_error();

inline Ctx* as_ctx(lq_ctx* c) { return static_cast<Ctx*>(c); }

// stream-ordered scratch buffer (cudaMallocAsync pool; no host synchronisation after warm-up)
struct DevBuf {
    Ctx* ctx = nullptr;
    void* p = nullptr;
    cudaStream_t s = nullptr;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() { release(); }
    int alloc(Ctx* c, size_t bytes, cudaStream_t stream = nullptr) {
        release();
        ctx = c;
        s = stream ? stream : c->stream;
        if (bytes == 0) bytes = 16;
        LQ_CUDA(c, cudaMallocAsync(&p, bytes, s));
        return LQ_OK;
    }
    void release() {
        if (p) cudaFreeAsync(p, s);
        p = nullptr;
    }
    template <typename T>
    T* as() const {
        return static_cast<T*>(p);
    }
};

}  // namespace lq

// K3 launch glue: streaming Householder least squares (stream_qr.cuh) for n <= 64, nrhs <= 32.
#include "../../include/linalg_b200.h"
#include "ops.cuh"
#include "stream_qr.cuh"
#include "lstsq_tile.cuh"

namespace lq {

bool lstsq_stream_kernel_supported(int m, int n, int nrhs) {
    return n >= 1 && n <= 64 && nrhs >= 1 && nrhs <= 32 && m >= n;
}

// rows per streamed block = RPT * WARPS = 16 * 4.  Taller blocks mean fewer column steps per system (every step pays the
// publish -> dots -> barrier -> norm / reciprocal chain once, whatever the block height).
int lstsq_stream_kernel_launch(Ctx* c, cudaStream_t st, const double* A, const double* B, long long batch, int m, int n,
                               int nrhs, double* X, int* info) {
    if (!lstsq_stream_kernel_supported(m, n, nrhs)) return LQ_ERR_UNSUPPORTED;
    constexpr int RPT = 16, WARPS = 4;
    const size_t smem = StreamCfg<3, RPT, WARPS>::smem_doubles(n) * sizeof(double);
    return launch<lstsq_stream_kernel<RPT, WARPS>>(c, batch, WARPS * 32, smem, st, c->max_smem, A, B, X, info, m, n, nrhs);
}

// ---- round 2: one warp per system, block reflectors on DMMA (lstsq_tile.cuh); n <= 64, nrhs <= 16
bool lstsq_tile_kernel_supported(int m, int n, int nrhs) {
    return n >= 1 && n <= 8 * LsTile::NCB && nrhs >= 1 && nrhs <= 8 * LsTile::NRT && m >= n;
}

int lstsq_tile_kernel_launch(Ctx* c, cudaStream_t st, const double* A, const double* B, long long batch, int m, int n,
                             int nrhs, double* X, int* info, int info_mode) {
    if (!lstsq_tile_kernel_supported(m, n, nrhs)) return LQ_ERR_UNSUPPORTED;
    // two 4-warp CTAs per SM: 17.4 ms (8 x 1: 17.8, 7 x 1: 19.9)
    constexpr int WARPS = 4;
    const size_t smem = (size_t)WARPS * LsTile::WARP_DOUBLES * sizeof(double);
    return launch<lstsq_tile_kernel<WARPS, 2>>(c, (batch + WARPS - 1) / WARPS, WARPS * 32, smem, st, (int)smem, A, B, X, info,
                                               batch, m, n, nrhs, info_mode);
}

}  // namespace lq

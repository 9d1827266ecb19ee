"""Host-pointer entry points on paths the Python API does not take: a null info pointer, an empty batch, and the
per-matrix route of householder_qr_batched over several matrices.

Each batched dispatcher either launches one kernel for the whole batch or runs the single-matrix path matrix by matrix;
its host-pointer entry point pipelines the first kind over two lanes and runs the second on the context stream.  Every
case below uses one shape on each side of that choice (the boundaries of ``test_gpu_routes``) and compares the host
entry point with the device entry point: the same bits and the same number of kernel launches.
"""
import numpy as np
import pytest

from test_gpu_routes import boundary, counted

pytestmark = pytest.mark.gpu

SIDES = [0, 1]   # 0: last shape of the one-launch route, 1: first shape of the per-matrix route


@pytest.fixture(scope="module")
def smem(ctx):
    return ctx.props()["max_smem"]


def _ptr(a):
    return a.ctypes.data


# host entry point, device entry point, boundary family; the device form of lq_lstsq_householder_batched has no info
NULL_INFO_LS = [
    ("lq_lstsq_householder_batched", "lq_lstsq_householder_batched_dev", "hh_ls"),
    ("lq_lstsq_householder_batched_info", "lq_lstsq_householder_batched_info_dev", "hh_ls"),
    ("lq_lstsq_mgs_batched", "lq_lstsq_mgs_batched_dev", "mgs_ls"),
]


@pytest.mark.parametrize("side", SIDES)
@pytest.mark.parametrize("host,dev,family", NULL_INFO_LS, ids=[h for h, _, _ in NULL_INFO_LS])
def test_least_squares_null_info(ctx, smem, host, dev, family, side):
    """Without info the host entry point gives the device entry point's X and launches the same kernels (the blocked
    Householder route skips its singularity report in both)."""
    m, n, k = boundary(family, smem)[side]
    nb = 3
    rng = np.random.default_rng(m + side)
    A, B = rng.standard_normal((nb, m, n)), rng.standard_normal((nb, m, k))
    info = () if host == "lq_lstsq_householder_batched" else (None,)
    dA, dB, dX = ctx.upload(A), ctx.upload(B), ctx.alloc(8 * nb * n * k)
    _, nl_dev = counted(ctx, ctx.call, dev, dA.ptr, dB.ptr, nb, m, n, k, dX.ptr, *info)
    X = np.full((nb, n, k), np.nan)
    _, nl_host = counted(ctx, ctx.call, host, _ptr(A), _ptr(B), nb, m, n, k, _ptr(X), *info)
    assert np.array_equal(X, ctx.download(dX, (nb, n, k)))
    assert nl_host == nl_dev, (nl_host, nl_dev)
    assert (nl_dev == 1) == (side == 0), nl_dev


@pytest.mark.parametrize("side", SIDES)
def test_mgs_qr_batched_null_info(ctx, smem, side):
    """qr_batched without info: the device entry point's Q and R, the same launches."""
    m, n = boundary("mgs_square", smem)[side]
    nb = 3
    A = np.random.default_rng(n).standard_normal((nb, m, n))
    dA, dQ, dR = ctx.upload(A), ctx.alloc(A.nbytes), ctx.alloc(8 * nb * n * n)
    _, nl_dev = counted(ctx, ctx.call, "lq_mgs_qr_batched_dev", dA.ptr, nb, m, n, 0, dQ.ptr, dR.ptr, None)
    Q, R = np.full(A.shape, np.nan), np.full((nb, n, n), np.nan)
    _, nl_host = counted(ctx, ctx.call, "lq_mgs_qr_batched", _ptr(A), nb, m, n, 0, _ptr(Q), _ptr(R), None)
    assert np.array_equal(Q, ctx.download(dQ, A.shape)) and np.array_equal(R, ctx.download(dR, R.shape))
    assert nl_host == nl_dev, (nl_host, nl_dev)


EMPTY = [
    ("lq_householder_qr_batched", "hh_square", lambda m, n, k: (None, 0, m, n, None, None)),
    ("lq_mgs_qr_batched", "mgs_square", lambda m, n, k: (None, 0, m, n, 0, None, None, None)),
    ("lq_lstsq_householder_batched", "hh_ls", lambda m, n, k: (None, None, 0, m, n, k, None)),
    ("lq_lstsq_householder_batched_info", "hh_ls", lambda m, n, k: (None, None, 0, m, n, k, None, None)),
    ("lq_lstsq_mgs_batched", "mgs_ls", lambda m, n, k: (None, None, 0, m, n, k, None, None)),
    ("lq_svd_gram_batched", "svd", lambda m, n, k: (None, 0, m, n, 1e-12, None, None, None, None)),
]


@pytest.mark.parametrize("side", SIDES)
@pytest.mark.parametrize("name,family,args", EMPTY, ids=[e[0] for e in EMPTY])
def test_empty_batch_launches_nothing(ctx, smem, name, family, args, side):
    """batch = 0 returns at once: no kernel, and no pointer is touched (all are null here)."""
    shape = ((4096, 32), (4097, 32))[side] if family == "svd" else boundary(family, smem)[side]  # svd_small_supported
    m, n, k = (*shape, 1)[:3]
    _, nl = counted(ctx, ctx.call, name, *args(m, n, k))
    assert nl == 0


def test_householder_qr_batched_per_matrix_route(ctx, smem):
    """The per-matrix route over 4 matrices calls lq_householder_qr_dev on the same three device buffers each time, so its
    graph cache runs plain launches, captures and replays.  Same bits and launches as the device entry point."""
    m, n = boundary("hh_square", smem)[1]
    nb = 4
    A = np.random.default_rng(n).standard_normal((nb, m, n))
    dA, dQ, dR = ctx.upload(A), ctx.alloc(A.nbytes), ctx.alloc(8 * nb * n * n)
    _, nl_dev = counted(ctx, ctx.call, "lq_householder_qr_batched_dev", dA.ptr, nb, m, n, dQ.ptr, dR.ptr, 0)
    Q, R = np.full(A.shape, np.nan), np.full((nb, n, n), np.nan)
    _, nl_host = counted(ctx, ctx.call, "lq_householder_qr_batched", _ptr(A), nb, m, n, _ptr(Q), _ptr(R))
    assert np.array_equal(Q, ctx.download(dQ, A.shape)) and np.array_equal(R, ctx.download(dR, R.shape))
    assert nl_host == nl_dev > nb, (nl_host, nl_dev)

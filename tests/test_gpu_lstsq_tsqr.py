"""least_squares_tsqr / lq_lstsq_tsqr*: tall-skinny least squares on the CholeskyQR2 pipeline, its Householder fallbacks,
and the row-sharded form over NCCL with two ranks.

Routes of one GPU (tsqr.cu, lstsq_tsqr_local):
- "fused":  n <= 128, m >= 4n, even n, nrhs <= 32, m >= 1024: pass 2 forms [G2 | C] = Q1^T [Q1 | B] in the strip SYRK kernel
  (an odd nrhs is padded to even);
- "gemm":   the other CholeskyQR2 shapes: SYRK or GEMM Gram matrix and a TN GEMM for Q1^T B;
- "householder": m < 4n, n > 128, an ill-conditioned A (cond^2 estimate >= 1e10) or TSQR_HOUSEHOLDER: exactly the route of
  least_squares_householder_qr, so the result is bitwise that function's.
"""
import os
import socket
import sys

import numpy as np
import pytest

import linalg_b200 as lb

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def route(m, n, k):
    if n > 128 or m < 4 * n:
        return "householder"
    return "fused" if (n % 2 == 0 and k <= 32 and m >= 1024) else "gemm"


def lapack(A, B):
    return np.linalg.lstsq(A, B, rcond=None)[0]


def rel(X, Xo):
    return np.max(np.abs(X - Xo)) / np.max(np.abs(Xo))


def resid(A, X, B):
    return np.linalg.norm(A @ X - B)


def backward_error(A, X, B):
    """max over the right-hand sides of ||A^T r|| / (||A|| (||A|| ||x|| + ||r||)), r = A x - b"""
    A2 = np.linalg.norm(A, 2)
    X, B = X.reshape(X.shape[0], -1), B.reshape(B.shape[0], -1)
    R = A @ X - B
    num = np.linalg.norm(A.T @ R, axis=0)
    return np.max(num / (A2 * (A2 * np.linalg.norm(X, axis=0) + np.linalg.norm(R, axis=0))))


def check_parity(A, B, X, label):
    Xo = lapack(A, B)
    assert X.shape == Xo.shape, label
    assert rel(X, Xo) <= 1e-10, (label, rel(X, Xo))
    ro = resid(A, Xo, B)
    assert abs(resid(A, X, B) - ro) <= 1e-10 * ro, (label, resid(A, X, B), ro)


# ----------------------------------------------------------------------------- host-side contract (no GPU touched)
def test_shape_errors_and_empty_results():
    with pytest.raises(ValueError):
        lb.least_squares_tsqr(np.zeros((3, 5)), np.zeros(3))
    with pytest.raises(ValueError):
        lb.least_squares_tsqr(np.zeros((8, 2)), np.zeros(7))
    with pytest.raises(ValueError):
        lb.least_squares_tsqr(np.zeros((8, 2)), np.zeros((8, 2, 1)))
    with pytest.raises(ValueError):
        lb.least_squares_tsqr(np.zeros(8), np.zeros(8))
    assert lb.least_squares_tsqr(np.zeros((8, 0)), np.zeros(8)).shape == (0,)
    assert lb.least_squares_tsqr(np.zeros((8, 3)), np.zeros((8, 0))).shape == (3, 0)
    assert "least_squares_tsqr" in lb.__all__


# ----------------------------------------------------------------------------- parity at 2^16 x 128
@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 16, 32, 33], ids=["vector", "k16", "k32", "k33"])
def test_parity_gaussian(ctx, k):
    m, n = 1 << 16, 128
    rng = np.random.default_rng(100 + k)
    A = rng.standard_normal((m, n))
    b = rng.standard_normal(m) if k == 1 else rng.standard_normal((m, k))
    A0, b0 = A.copy(), b.copy()
    x = lb.least_squares_tsqr(A, b, ctx=ctx)
    assert np.array_equal(A, A0) and np.array_equal(b, b0)  # inputs are never mutated
    assert x.shape == ((n,) if k == 1 else (n, k))
    check_parity(A, b, x, k)
    # a consistent system (zero residual)
    x0 = rng.standard_normal((n,) if k == 1 else (n, k))
    xc = lb.least_squares_tsqr(A, A @ x0, ctx=ctx)
    assert np.linalg.norm(xc - x0) <= 1e-12 * np.linalg.norm(x0), np.linalg.norm(xc - x0) / np.linalg.norm(x0)


# ----------------------------------------------------------------------------- route boundaries
ROUTE_CASES = [
    ("m_4n_minus_1", (4 * 64 - 1, 64, 4)),
    ("m_4n", (4 * 64, 64, 4)),
    ("odd_n", (5000, 63, 8)),
    ("n1", (5000, 1, 3)),
    ("n128_m_not_16", (4096 + 5, 128, 8)),
    ("n129", (5000, 129, 4)),
    ("m_not_16", (2000 + 7, 64, 2)),
    ("m_below_1024", (1000, 32, 6)),
    ("odd_k", (3001, 40, 5)),
    ("k_over_32", (3000, 40, 40)),
]


@pytest.mark.gpu
@pytest.mark.parametrize("label,shape", ROUTE_CASES, ids=[c[0] for c in ROUTE_CASES])
def test_route_boundaries(ctx, label, shape):
    m, n, k = shape
    rng = np.random.default_rng(m + 7 * n + k)
    A = rng.standard_normal((m, n))
    B = rng.standard_normal((m, k))
    X = lb.least_squares_tsqr(A, B, ctx=ctx)
    check_parity(A, B, X, label)
    Xh = lb.least_squares_householder_qr(A, B, ctx=ctx)
    # the Householder route is exactly least_squares_householder_qr; the CholeskyQR2 routes are a different computation
    assert np.array_equal(X, Xh) == (route(m, n, k) == "householder"), (label, route(m, n, k))


@pytest.mark.gpu
def test_householder_option_takes_the_householder_route(ctx):
    rng = np.random.default_rng(5)
    A, B = rng.standard_normal((4096, 64)), rng.standard_normal((4096, 4))
    ctx.set_option("TSQR_HOUSEHOLDER", True)
    try:
        X = lb.least_squares_tsqr(A, B, ctx=ctx)
    finally:
        ctx.set_option("TSQR_HOUSEHOLDER", False)
    assert np.array_equal(X, lb.least_squares_householder_qr(A, B, ctx=ctx))
    assert not np.array_equal(X, lb.least_squares_tsqr(A, B, ctx=ctx))


@pytest.mark.gpu
def test_device_entry_point_and_info(ctx):
    m, n, k = 8192, 96, 12
    rng = np.random.default_rng(11)
    A, B = rng.standard_normal((m, n)), rng.standard_normal((m, k))
    dA, dB, dX, dI = ctx.upload(A), ctx.upload(B), ctx.alloc(8 * n * k), ctx.upload(np.full(1, -1, np.int32))
    ctx.call("lq_lstsq_tsqr_dev", dA.ptr, m, n, dB.ptr, k, dX.ptr, dI.ptr)
    assert ctx.download(dI, (1,), dtype=np.int32)[0] == 0
    assert np.array_equal(ctx.download(dX, (n, k)), lb.least_squares_tsqr(A, B, ctx=ctx))
    with pytest.raises(ValueError):
        ctx.call("lq_lstsq_tsqr_dev", dA.ptr, n - 1, n, dB.ptr, k, dX.ptr, dI.ptr)


# ----------------------------------------------------------------------------- ill-conditioned and singular input
@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(1 << 14, 64, 3), (1 << 14, 128, 1)], ids=["n64", "n128"])
def test_ill_conditioned_declines_the_fast_path(ctx, shape):
    m, n, k = shape
    rng = np.random.default_rng(n + k)
    A = rng.standard_normal((m, n)) * np.logspace(0.0, -9.0, n)[None, :]  # cond ~ 1e9
    B = rng.standard_normal((m, k))
    X = lb.least_squares_tsqr(A, B, ctx=ctx)
    if n <= 64:
        # CholeskyQR2 declined: bitwise the Householder route (for n > 64 that route factors panels taller than 16 x 512 rows
        # with atomic partial sums, not bitwise reproducible; the backward error below is what CholeskyQR2 cannot reach here)
        assert np.array_equal(X, lb.least_squares_householder_qr(A, B, ctx=ctx))
    assert backward_error(A, X, B) <= 1e-12, backward_error(A, X, B)
    ro = resid(A, lapack(A, B), B)
    assert abs(resid(A, X, B) - ro) <= 1e-10 * ro


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(4096, 32), (300, 100), (5000, 130)], ids=["cholqr2_declines", "householder", "wide"])
def test_exactly_zero_column_raises_like_householder(ctx, shape):
    m, n = shape
    rng = np.random.default_rng(m)
    A = rng.standard_normal((m, n))
    A[:, 5] = 0.0
    b = rng.standard_normal(m)
    with pytest.raises(np.linalg.LinAlgError, match="Singular matrix"):
        lb.least_squares_householder_qr(A, b, ctx=ctx)
    with pytest.raises(np.linalg.LinAlgError, match="Singular matrix"):
        lb.least_squares_tsqr(A, b, ctx=ctx)


# ----------------------------------------------------------------------------- power-of-two scaling
SCALING_CASES = [("fused", (4096, 64, 8)), ("fused_odd_k", (4096, 64, 1)), ("gemm", (3000, 63, 5)),
                 ("householder", (200, 64, 3))]


@pytest.mark.gpu
@pytest.mark.parametrize("label,shape", SCALING_CASES, ids=[c[0] for c in SCALING_CASES])
def test_power_of_two_scaling(ctx, label, shape):
    """X(4^j A, 4^jt B) = 4^(jt - j) X(A, B) bit for bit over the exponent range of the tall-skinny family."""
    from test_gpu_scaling import NORM_MAX_LOG2, log2, qr_js, sc

    m, n, k = shape
    assert route(m, n, k) == label.split("_")[0]
    rng = np.random.default_rng(m + n + k)
    A, B = rng.standard_normal((m, n)), rng.standard_normal((m, k))
    X0 = lb.least_squares_tsqr(A, B, ctx=ctx)
    js = qr_js(A)
    bmax = log2(np.max(np.linalg.norm(B, axis=0)))
    for j in js:
        for jt in sorted({j, -j, 0}):
            if 2 * jt + bmax > NORM_MAX_LOG2:
                continue
            X = lb.least_squares_tsqr(sc(A, j), sc(B, jt), ctx=ctx)
            assert np.array_equal(X, sc(X0, jt - j)), (label, j, jt, np.max(np.abs(X - sc(X0, jt - j))))
        if j in (js[0], js[-1]):
            check_parity(sc(A, j), sc(B, j), lb.least_squares_tsqr(sc(A, j), sc(B, j), ctx=ctx), (label, j))


# ----------------------------------------------------------------------------- two ranks
def _ngpu():
    import ctypes

    from linalg_b200 import _native

    n = ctypes.c_int(0)
    _native.load_library().lq_device_count(ctypes.byref(n))
    return n.value


SHARDED = {
    # name: (rows, n, nrhs, householder tree forced, column scaling decades, uneven split)
    "gaussian": (1 << 16, 96, 8, False, 0.0, False),
    "uneven_shards": ((1 << 13) + 517, 96, 8, False, 0.0, True),
    "householder_tree": (1 << 14, 96, 8, True, 0.0, False),
    "ill_conditioned": (1 << 14, 96, 8, False, 9.0, False),
    "ill_conditioned_too_wide": (1 << 14, 128, 4, False, 9.0, False),  # tree of [A | B] needs n + nrhs <= 128
}


def _sharded_case(name):
    m, n, k, _, span, _ = SHARDED[name]
    rng = np.random.default_rng(len(name))
    A = rng.standard_normal((m, n))
    if span:
        A = A * np.logspace(0.0, -span, n)[None, :]
    return A, rng.standard_normal((m, k))


def _sharded_bounds(name, rank, world):
    m, uneven = SHARDED[name][0], SHARDED[name][5]
    if uneven:
        cut = (3 * m) // 8
        return (0, cut) if rank == 0 else (cut, m)
    from linalg_b200.utils import shard_bounds

    return shard_bounds(m, world, rank)


def _worker(rank, world, port, outdir):
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1",
                      MASTER_PORT=str(port), LINALG_B200_DEVICE=str(rank))
    sys.path.insert(0, ROOT)
    import linalg_b200 as lbw
    from linalg_b200 import dist as d

    info = d.init_control_plane("gloo")
    ctx = lbw.Context(rank)
    d.init_comm(ctx, info)
    for name, (_, n, k, tree, _, _) in SHARDED.items():
        A, B = _sharded_case(name)
        lo, hi = _sharded_bounds(name, rank, world)
        dA, dB = ctx.upload(np.ascontiguousarray(A[lo:hi])), ctx.upload(np.ascontiguousarray(B[lo:hi]))
        dX, dI = ctx.alloc(8 * n * k), ctx.upload(np.full(1, -1, np.int32))
        ctx.set_option("TSQR_HOUSEHOLDER", tree)
        err = ""
        try:
            ctx.call("lq_lstsq_tsqr_sharded_dev", dA.ptr, hi - lo, n, dB.ptr, k, dX.ptr, dI.ptr)
            X, inf = ctx.download(dX, (n, k)), ctx.download(dI, (1,), dtype=np.int32)
        except (ValueError, NotImplementedError) as exc:
            err, X, inf = f"{type(exc).__name__}: {exc}", np.zeros((n, k)), np.full(1, -1, np.int32)
        ctx.set_option("TSQR_HOUSEHOLDER", False)
        np.savez(os.path.join(outdir, f"{name}_r{rank}.npz"), lo=lo, hi=hi, X=X, info=inf, err=err)
        for buf in (dA, dB, dX, dI):
            buf.free()
    d.barrier()
    ctx.call("lq_comm_destroy")
    d.shutdown_control_plane()


@pytest.mark.gpu
def test_sharded_lstsq_two_ranks(tmp_path):
    if _ngpu() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp

    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    for name in SHARDED:
        A, B = _sharded_case(name)
        z = [np.load(tmp_path / f"{name}_r{r}.npz") for r in range(2)]
        assert int(z[0]["hi"]) == int(z[1]["lo"]) and int(z[1]["hi"]) == A.shape[0], name
        err = [str(z[r]["err"]) for r in range(2)]
        if name == "ill_conditioned_too_wide":
            assert err[0] and err[0] == err[1] and "n + nrhs" in err[0], err
            continue
        assert err == ["", ""], (name, err)
        assert np.array_equal(z[0]["X"], z[1]["X"]) and np.array_equal(z[0]["info"], z[1]["info"]), name  # replicated
        assert int(z[0]["info"][0]) == 0, name
        X = z[0]["X"]
        if name == "ill_conditioned":
            assert backward_error(A, X, B) <= 1e-12, (name, backward_error(A, X, B))
            ro = resid(A, lapack(A, B), B)
            assert abs(resid(A, X, B) - ro) <= 1e-10 * ro, name
        else:
            check_parity(A, B, X, name)

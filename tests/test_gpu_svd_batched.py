"""svd_batched: the A^T A economy SVD of every matrix of a batch.

Matrix i of the result is ``svd(A[i], tol)``.  The route depends on the shape alone (``svd_small_supported``, which
``svd_batched_stream`` in ``api_batched.cu`` and the host-pointer entry point in ``api_host.cu`` both call): n <= 32 and
m <= 4096 after transposition run the warp-per-matrix kernel (one launch per call or per host-pipeline chunk), every
other shape runs the single-matrix pipeline matrix by matrix and is bitwise ``svd(A[i])``.  Each matrix is held to the
bounds of ``svd`` against LAPACK (``svd_errors`` of ``test_gpu_tallskinny_routes``).
"""
import numpy as np
import pytest

import linalg_b200 as lb
from linalg_b200 import _native as nat
from oracle import linalg_oracle as orc
from test_gpu_routes import U64, counted
from test_gpu_scaling import gram_js, same, sc
from test_gpu_tallskinny_routes import (C_SVD, C_SVD_RECON, ORTH, REL, SVD_SPECTRA, assert_within, conditioned, svd_errors,
                                        svd_input)

N_MAX = 32        # SvdSmall::NMAX
M_SMALL = 4096    # SvdSmall::M_SMALL


def route(m, n):
    m, n = max(m, n), min(m, n)
    return "kernel" if n <= N_MAX and m <= M_SMALL else "per_matrix"


# ----------------------------------------------------------------------------- host only
def test_svd_batched_is_exported():
    assert "svd_batched" in lb.__all__ and callable(lb.svd_batched)


@pytest.fixture
def no_device(monkeypatch):
    def boom(*a, **k):
        raise AssertionError("device work before the argument check")

    monkeypatch.setattr(nat, "default_context", boom)
    monkeypatch.setattr(nat, "device_context", boom)


def test_argument_errors(no_device):
    for bad in (np.ones((4, 4)), np.ones((2, 2, 3, 3)), np.ones(3)):
        with pytest.raises(ValueError):
            lb.svd_batched(bad)
    A = np.ones((2, 5, 3))
    good = (np.empty((2, 5, 3)), np.empty((2, 3)), np.empty((2, 3, 3)))
    for i, bad in enumerate([np.empty((2, 5, 4)), np.empty((2, 3), dtype=np.float32), np.empty((2, 3, 3))[:, :, ::-1]]):
        out = list(good)
        out[i] = bad
        with pytest.raises(ValueError):
            lb.svd_batched(A, out=tuple(out))
    with pytest.raises(ValueError):
        lb.svd_batched(A, ctx=object(), devices=[0])


@pytest.mark.parametrize("shape", [(0, 3, 2), (0, 2, 3), (2, 0, 5), (2, 5, 0), (3, 0, 0)])
def test_empty_shapes(no_device, shape):
    b, m, n = shape
    k = min(m, n)
    U, s, Vt = lb.svd_batched(np.zeros(shape))
    assert U.shape == (b, m, k) and s.shape == (b, k) and Vt.shape == (b, k, n)


def test_route_is_the_shape_alone():
    assert [route(*s) for s in [(32, 32), (32, 1), (M_SMALL, 32), (16, 32), (M_SMALL + 1, 32), (40, 33), (33, 40)]] == \
        ["kernel"] * 4 + ["per_matrix"] * 3


# ----------------------------------------------------------------------------- accuracy
ACC_SHAPES = [(32, 32), (32, 1), (17, 5), (256, 16), (M_SMALL, 32), (M_SMALL + 1, 32), (40, 33), (16, 32)]


def check_matrix(A, U, s, Vt, cluster, label):
    """svd's bounds against LAPACK; a wide matrix is checked as the transposed decomposition (svd.py:37-39).  The bounds
    scale with m, and a few rows leave the reference algorithm itself (oracle.svd_gram, LAPACK's eigh of A^T A) slightly
    above them on some inputs (17 x 5 at kappa 1e4: 1.03 x the eigenvector bound): a check is met within its bound or
    within twice the reference algorithm's error on the same matrix."""
    if A.shape[0] < A.shape[1]:
        A, U, Vt = A.T, Vt.T, U.T
    _, sigma, VtL = np.linalg.svd(A, full_matrices=False)
    assert np.all(np.diff(s) <= 0), label
    errs = svd_errors(A, U, s, Vt, sigma, VtL.T, cluster)
    ref = svd_errors(A, *orc.svd_gram(A), sigma, VtL.T, cluster)
    if A.shape[1] == 1:   # one column: no gap, the vector bound is 0 / 0; V = +-1 is held by v_orth
        errs.pop("vector", None)
    assert_within(label, **{k: (e, max(b, 2 * ref[k][0])) for k, (e, b) in errs.items()})


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ACC_SHAPES, ids=lambda s: f"{s[0]}x{s[1]}")
def test_accuracy_per_matrix(ctx, shape):
    """Every spectrum of the single-matrix SVD tests in one batch (gaussian, kappa 1e2 / 1e4 / 1e6, a cluster of equal
    values, scaled input), two matrices each; each matrix meets svd's bounds."""
    m, n = shape
    tall = (max(m, n), min(m, n))
    rng = np.random.default_rng(m * 64 + n)
    mats, clusters = [], []
    for spectrum in SVD_SPECTRA:
        for _ in range(2):
            X, cl = svd_input(spectrum, *tall, rng)
            mats.append(X if m >= n else X.T)
            clusters.append(cl)
    A = np.stack(mats)
    U, s, Vt = lb.svd_batched(A, ctx=ctx)
    k = min(m, n)
    assert U.shape == (len(A), m, k) and s.shape == (len(A), k) and Vt.shape == (len(A), k, n)
    for i in range(len(A)):
        check_matrix(A[i], U[i], s[i], Vt[i], clusters[i], f"{route(m, n)} {SVD_SPECTRA[i // 2]} #{i}")


def sign_match(U, Uo):
    return np.where(np.sum(U * Uo, axis=0) < 0, -1.0, 1.0)


@pytest.mark.gpu
def test_reference_parity(ctx):
    """The reference's own seeded cases (tests/test_svd.py: (8, 5), (20, 20), (50, 10), (12, 7), (30, 15)), each in a
    batch with Gaussian matrices of its shape, and a batch of Gaussian 32 x 32 matrices, against the reference algorithm
    (oracle.svd_gram, matrix by matrix) at the reference's tolerances."""
    cases = [((8, 5), 13), ((20, 20), 40), ((50, 10), 60), ((12, 7), 55), ((30, 15), 135), ((32, 32), None)]
    for (m, n), seed in cases:
        rng = np.random.default_rng(m * n)
        A = rng.standard_normal((6, m, n))
        if seed is not None:
            A[2] = np.random.default_rng(seed=seed).standard_normal(size=(m, n))
        U, s, Vt = lb.svd_batched(A, ctx=ctx)
        for i in range(len(A)):
            Uo, so, Vto = orc.svd_gram(A[i])
            np.testing.assert_allclose(s[i], so, rtol=1e-10, atol=1e-12)
            sg = sign_match(U[i], Uo)
            assert np.max(np.abs(U[i] * sg - Uo)) <= 1e-8, (m, n, i)
            assert np.max(np.abs(Vt[i] * sg[:, None] - Vto)) <= 1e-8, (m, n, i)


# ----------------------------------------------------------------------------- routes
@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(M_SMALL + 1, 32), (40, 33), (33, 40)], ids=lambda s: f"{s[0]}x{s[1]}")
def test_per_matrix_route_is_svd(ctx, shape):
    A = np.random.default_rng(sum(shape)).standard_normal((3,) + shape)
    assert route(*shape) == "per_matrix"
    U, s, Vt = lb.svd_batched(A, ctx=ctx)
    for i in range(len(A)):
        U1, s1, Vt1 = lb.svd(A[i], ctx=ctx)
        same(f"U {i}", U[i], U1)
        same(f"s {i}", s[i], s1)
        same(f"Vt {i}", Vt[i], Vt1)


def run_dev(ctx, A, tol=1e-12):
    """lq_svd_gram_batched_dev on A (batch, m, n), m >= n: (U, s, Vt, rank) and the kernels it launched."""
    b, m, n = A.shape
    dA, dU, ds, dV, dr = ctx.upload(A), ctx.alloc(8 * b * m * n), ctx.alloc(8 * b * n), ctx.alloc(8 * b * n * n), ctx.alloc(4 * b)
    _, nl = counted(ctx, ctx.call, "lq_svd_gram_batched_dev", dA.ptr, b, m, n, float(tol), dU.ptr, ds.ptr, dV.ptr, dr.ptr)
    out = (ctx.download(dU, (b, m, n)), ctx.download(ds, (b, n)), ctx.download(dV, (b, n, n)),
           ctx.download(dr, (b,), dtype=np.int32))
    return out, nl


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(32, 32), (32, 1), (M_SMALL, 32), (M_SMALL + 1, 32)], ids=lambda s: f"{s[0]}x{s[1]}")
def test_launches_per_call(ctx, shape):
    """The kernel route is one launch whatever the batch size; the per-matrix route launches per matrix.  The host entry
    point gives the device entry point's result."""
    rng = np.random.default_rng(shape[0])
    counts = []
    for b in (1, 5):
        A = rng.standard_normal((b,) + shape)
        (U, s, Vt, r), nl = run_dev(ctx, A)
        counts.append(nl)
        U2, s2, Vt2 = lb.svd_batched(A, ctx=ctx)
        same("U", U, U2)
        same("s", s, s2)
        same("Vt", Vt, Vt2)
        assert np.all(r == shape[1])
    if route(*shape) == "kernel":
        assert counts == [1, 1], counts
    else:
        assert counts[1] == 5 * counts[0] and counts[0] > 1, counts


# ----------------------------------------------------------------------------- invariance
@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(32, 32), (17, 5), (256, 16)], ids=lambda s: f"{s[0]}x{s[1]}")
def test_batch_size_and_position_invariance(ctx, shape):
    rng = np.random.default_rng(7 + shape[1])
    X = rng.standard_normal(shape)
    ref = lb.svd_batched(X[None], ctx=ctx)
    for b, pos in [(1, 0), (7, 3), (7, 6), (4099, 0), (4099, 2050), (4099, 4098)]:
        A = rng.standard_normal((b,) + shape)
        A[pos] = X
        for run in range(2 if b == 7 else 1):
            got = lb.svd_batched(A, ctx=ctx)
            for g, r, name in zip(got, ref, "U s Vt".split()):
                same(f"{name} b={b} pos={pos} run={run}", g[pos], r[0])


@pytest.mark.gpu
@pytest.mark.parametrize("devices", [[0], [0, 1]], ids=["one", "two"])
def test_devices_kwarg(ctx, devices):
    if len(devices) > nat.device_count():
        pytest.skip(f"devices={devices} needs {len(devices)} visible GPUs")
    A = np.random.default_rng(3).standard_normal((37, 32, 32))
    A[5, :, 20:] = 0.0   # rank deficient: the completion runs after the split
    ref = lb.svd_batched(A, ctx=ctx, seed=4)
    got = lb.svd_batched(A, devices=devices, seed=4)
    for g, r, name in zip(got, ref, "U s Vt".split()):
        same(f"{name} devices={devices}", g, r)


# ----------------------------------------------------------------------------- scaling
@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(32, 32), (256, 16), (17, 5)], ids=lambda s: f"{s[0]}x{s[1]}")
def test_power_of_two_scaling(ctx, shape):
    """tol = 0: svd_batched(4^j A) = (U, 4^j s, Vt) bit for bit, for j across the range of the Gram-type sweeps."""
    rng = np.random.default_rng(shape[0] + 1)
    A = np.stack([rng.standard_normal(shape), conditioned(rng, *shape, 1e4), rng.standard_normal(shape)])
    U0, s0, Vt0 = lb.svd_batched(A, 0.0, ctx=ctx)
    dmax = max(np.linalg.svd(a, compute_uv=False)[0] ** 2 for a in A)
    for j in gram_js(dmax):
        U, s, Vt = lb.svd_batched(sc(A, j), 0.0, ctx=ctx)
        same(f"U j={j}", U, U0)
        same(f"s j={j}", s, sc(s0, j))
        same(f"Vt j={j}", Vt, Vt0)


# ----------------------------------------------------------------------------- rank deficiency
def rank_batch(m, n, rng):
    """Full-rank matrices between matrices with exactly zero columns (rank 0, 1, n - 1)."""
    ranks = [n, 0, n, 1, n - 1, n]
    A = rng.standard_normal((len(ranks), m, n))
    for i, r in enumerate(ranks):
        A[i, :, r:] = 0.0
    return A, ranks


def check_completion(A, U, s, Vt, r, label):
    """The first r columns of U meet svd's bounds; the completion U[:, r:] is orthonormal, and orthogonal to U_r within
    U_r's own bound (as test_svd_tol_cuts_small_singular_values holds the single path)."""
    m, n = A.shape
    _, sigma, VtL = np.linalg.svd(A, full_matrices=False)
    if r:
        assert_within(label, **svd_errors(A, U, s, Vt, sigma, VtL.T, r=r))
    if r < n:
        Uc = U[:, r:]
        assert np.max(np.abs(Uc.T @ Uc - np.eye(n - r))) <= ORTH, label
        if r:
            assert np.max(np.abs(U[:, :r].T @ Uc)) <= C_SVD * m * U64 * (sigma[0] / s[r - 1]) ** 2, label


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(32, 32), (40, 8), (M_SMALL + 1, 4)], ids=lambda s: f"{s[0]}x{s[1]}")
def test_rank_deficient_completion(ctx, shape):
    """seed=None: the global RNG ends where a loop over svd leaves it, and the completed columns are the loop's up to sign.
    seed=k: the first r columns meet svd's bounds, the completion is orthonormal, reconstruction within svd's bound."""
    m, n = shape
    A, ranks = rank_batch(m, n, np.random.default_rng(m + n))
    np.random.seed(17)
    loop = [lb.svd(a, ctx=ctx) for a in A]
    after_loop = np.random.get_state()
    np.random.seed(17)
    U, s, Vt = lb.svd_batched(A, ctx=ctx)
    after_batch = np.random.get_state()
    assert after_loop[0] == after_batch[0] and np.array_equal(after_loop[1], after_batch[1]) and after_loop[2:] == after_batch[2:]
    for i, r in enumerate(ranks):
        assert int(np.sum(s[i] > 1e-12)) == r, (i, r)
        if r < n:
            Ul = loop[i][0]
            sg = sign_match(U[i][:, r:], Ul[:, r:])
            assert orc.rel_max_err(U[i][:, r:] * sg, Ul[:, r:]) <= REL, (i, r)
    U2, s2, Vt2 = lb.svd_batched(A, ctx=ctx, seed=11)
    same("s seeded", s2, s)
    for i, r in enumerate(ranks):
        check_completion(A[i], U2[i], s2[i], Vt2[i], r, f"seeded #{i}")
        assert np.linalg.norm(A[i] - (U2[i] * s2[i]) @ Vt2[i]) <= C_SVD_RECON * n * U64 * np.linalg.norm(A[i]), i
        if route(m, n) == "per_matrix":
            same(f"U seeded {i}", U2[i], lb.svd(A[i], ctx=ctx, seed=11)[0])


@pytest.mark.gpu
def test_tol_cut(ctx):
    """tol = 1e-3 on geometric spectra from 1 down to 1 / kappa (1e6 and 1e5 are cut, 1e2 keeps full rank): rank =
    #(sigma > tol) per matrix, U's first r columns meet svd's bounds, the completion is orthonormal."""
    m, n, tol = 64, 32, 1e-3
    rng = np.random.default_rng(64)
    A = np.stack([conditioned(rng, m, n, kappa) for kappa in (1e6, 1e2, 1e5)])
    U, s, Vt = lb.svd_batched(A, tol, ctx=ctx, seed=2)
    for i in range(len(A)):
        _, sigma, VtL = np.linalg.svd(A[i], full_matrices=False)
        r = int(np.sum(sigma > tol))
        assert int(np.sum(s[i] > tol)) == r
        check_completion(A[i], U[i], s[i], Vt[i], r, f"tol #{i}")


# ----------------------------------------------------------------------------- full size
@pytest.mark.gpu
def test_full_size_2_20_matrices(ctx):
    """2^20 x 32 x 32 through the device entry point: every output finite, s descending, rank 32; 4096 sampled matrices
    meet svd's bounds against LAPACK."""
    b, m, n = 1 << 20, 32, 32
    dA, dU, ds, dV, dr = ctx.alloc(8 * b * m * n), ctx.alloc(8 * b * m * n), ctx.alloc(8 * b * n), ctx.alloc(8 * b * n * n), ctx.alloc(4 * b)
    ctx.call("lq_random_normal_dev", dA.ptr, b * m * n, 2024)
    ctx.call("lq_svd_gram_batched_dev", dA.ptr, b, m, n, 1e-12, dU.ptr, ds.ptr, dV.ptr, dr.ptr)
    ctx.sync()
    s = ctx.download(ds, (b, n))
    assert np.all(np.isfinite(s)) and np.all(np.diff(s, axis=1) <= 0)
    assert np.all(ctx.download(dr, (b,), dtype=np.int32) == n)
    step = 1 << 14   # matrices per chunk of the finiteness check
    buf = np.empty((step, m, n))
    for buf_dev in (dU, dV):
        for lo in range(0, b, step):
            ctx.call("lq_memcpy_d2h", buf.ctypes.data, buf_dev.ptr + 8 * lo * m * n, buf.nbytes)
            ctx.sync()
            assert np.all(np.isfinite(buf)), lo
    idx = np.sort(np.random.default_rng(5).choice(b, 4096, replace=False))
    one = np.empty((m, n))
    for i in idx:
        got = []
        for dev in (dA, dU, dV):
            ctx.call("lq_memcpy_d2h", one.ctypes.data, dev.ptr + 8 * int(i) * m * n, one.nbytes)
            ctx.sync()
            got.append(one.copy())
        check_matrix(got[0], got[1], s[i], got[2], 0, f"full size #{i}")

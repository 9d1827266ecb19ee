"""Parity of the CUDA path (through the C ABI) with the oracle and the reference-generated golden
fixtures.  Bars (BASELINE.json north_star): Q, R elementwise relative 1e-10 under the reference's
sign convention; ||A - QR|| / ||A|| <= 1e-12; max|Q^T Q - I| <= 1e-12; least-squares solutions and
singular values relative 1e-10."""
import ctypes as C

import numpy as np
import pytest

import linalg_b200 as lb
from conftest import golden_cases
from oracle import linalg_oracle as orc

pytestmark = pytest.mark.gpu

REL = 1e-10
RESID = 1e-12
ORTH = 1e-12


def check_qr(A, Q, R, Qo, Ro, rel=REL, mgs=False):
    assert Q.shape == Qo.shape and R.shape == Ro.shape
    assert orc.rel_max_err(Q, Qo) <= rel, ("Q", orc.rel_max_err(Q, Qo))
    assert orc.rel_max_err(R, Ro) <= rel, ("R", orc.rel_max_err(R, Ro))
    assert np.all(np.tril(R, -1) == 0.0)
    if not mgs:  # one-sweep MGS loses orthogonality like the reference does; compared elementwise only
        assert orc.orth_error(Q) <= ORTH
    assert orc.qr_residual(A, Q, R) <= RESID


# ------------------------------------------------------------------ a1 Householder, golden fixtures
@pytest.mark.parametrize("name", golden_cases("hh"))
def test_householder_golden(ctx, golden, name):
    A = golden[f"hh/{name}/A"]
    Q, R = lb.householder_qr(A, ctx=ctx)
    Qo, Ro = golden[f"hh/{name}/Q"], golden[f"hh/{name}/R"]
    assert Q.shape == Qo.shape and R.shape == Ro.shape
    assert orc.rel_max_err(Q, Qo) <= REL and orc.rel_max_err(R, Ro) <= REL
    assert np.all(np.tril(R, -1) == 0.0)
    if name != "all_zero":
        assert orc.qr_residual(A, Q, R) <= RESID
    assert orc.orth_error(Q) <= ORTH


@pytest.mark.parametrize("name", golden_cases("mgs"))
def test_mgs_golden(ctx, golden, name):
    A = golden[f"mgs/{name}/A"]
    Q, R = lb.qr(A, ctx=ctx)
    check_qr(A, Q, R, golden[f"mgs/{name}/Q"], golden[f"mgs/{name}/R"], mgs=True)
    assert np.all(np.diag(R) > 0)


@pytest.mark.parametrize("name", golden_cases("mgs_reorth"))
def test_mgs_reorth_golden(ctx, golden, name):
    A = golden[f"mgs_reorth/{name}/A"]
    Q, R = lb.qr(A, reorth=True, ctx=ctx)
    # the reference returns the SECOND sweep's R (~I), so Q @ R != A by design (qr.py:46-47)
    assert orc.rel_max_err(Q, golden[f"mgs_reorth/{name}/Q"]) <= REL
    assert np.max(np.abs(R - golden[f"mgs_reorth/{name}/R"])) <= 1e-10
    assert orc.orth_error(Q) <= ORTH


def test_batched32_golden(ctx, golden):
    A = golden["batched32/A"]
    Q, R = lb.householder_qr_batched(A, ctx=ctx)
    assert orc.rel_max_err(Q, golden["batched32/Q_hh"]) <= REL and orc.rel_max_err(R, golden["batched32/R_hh"]) <= REL
    Q, R = lb.qr_batched(A, ctx=ctx)
    assert orc.rel_max_err(Q, golden["batched32/Q_mgs"]) <= REL and orc.rel_max_err(R, golden["batched32/R_mgs"]) <= REL


# ------------------------------------------------------------------ cfg2: batched 32x32
@pytest.mark.parametrize("batch", [1, 3, 5, 33, 1000])
def test_batched32_ragged_batches(ctx, batch):
    A = np.random.default_rng(100 + batch).standard_normal((batch, 32, 32))
    Q, R = lb.householder_qr_batched(A, ctx=ctx)
    Qo, Ro = orc.householder_qr_batched(A)
    for i in range(0, batch, max(1, batch // 16)):
        check_qr(A[i], Q[i], R[i], Qo[i], Ro[i])
    assert orc.rel_max_err(Q, Qo) <= REL and orc.rel_max_err(R, Ro) <= REL
    Q, R = lb.qr_batched(A, ctx=ctx)
    Qo, Ro = orc.mgs_qr_batched(A)
    assert orc.rel_max_err(Q, Qo) <= REL and orc.rel_max_err(R, Ro) <= REL
    Q, R = lb.qr_batched(A, reorth=True, ctx=ctx)
    Qo, Ro = orc.mgs_qr_batched(A, reorth=True)
    assert orc.rel_max_err(Q, Qo) <= REL and np.max(np.abs(R - Ro)) <= 1e-10


def test_batched32_empty_batch(ctx):
    Q, R = lb.householder_qr_batched(np.zeros((0, 32, 32)), ctx=ctx)
    assert Q.shape == (0, 32, 32) and R.shape == (0, 32, 32)


def test_batched32_special_matrices(ctx):
    """Skip branch (||x|| < 1e-12, qr.py:79-80), negative/zero pivots, identity, tiny and huge scales."""
    rng = np.random.default_rng(77)
    A = rng.standard_normal((12, 32, 32))
    A[0] = 0.0
    A[1] = np.eye(32)
    A[2] = -np.eye(32)
    A[3][:, 5] = 0.0
    A[4] = np.triu(A[4])
    A[5] *= 1e-6
    A[6] *= 1e6
    A[7][:, 0] = 0.0
    A[7][0, 0] = 0.0
    A[8] = np.tril(A[8])
    A[9][10:, :] = 0.0  # rank 10: later columns hit the skip branch after elimination (tiny norms)
    Q, R = lb.householder_qr_batched(A, ctx=ctx)
    Qo, Ro = orc.householder_qr_batched(A)
    for i in range(12):
        if i == 9:
            # rank-deficient: reflectors of the numerically-zero tail are rounding noise in the
            # reference too; only the invariants are meaningful
            assert orc.qr_residual(A[i], Q[i], R[i]) <= RESID and orc.orth_error(Q[i]) <= ORTH
            continue
        assert orc.rel_max_err(Q[i], Qo[i]) <= REL, i
        assert orc.rel_max_err(R[i], Ro[i]) <= REL, i
    assert np.all(np.tril(R, -1) == 0.0)


def test_batched32_device_resident_full_size(ctx):
    """2^20 matrices resident in HBM (BASELINE cfg2) through the _dev entry points: parity on a
    strided subsample, invariants on another, determinism across replicas of the same input."""
    uniq, reps = 1 << 14, 64
    batch = uniq * reps
    A = np.random.default_rng(2).standard_normal((uniq, 32, 32))
    per = A.nbytes
    dA, dQ, dR = ctx.alloc(per * reps), ctx.alloc(per * reps), ctx.alloc(per * reps)
    ctx.call("lq_memcpy_h2d", dA.ptr, A.ctypes.data, per)
    for r in range(1, reps):
        ctx.call("lq_memcpy_d2d", dA.ptr + r * per, dA.ptr, per)
    for which in ("hh", "mgs"):
        if which == "hh":
            ctx.call("lq_householder_qr_batched_dev", dA.ptr, batch, 32, 32, dQ.ptr, dR.ptr, 0)
        else:
            dI = ctx.alloc(4 * batch)
            ctx.call("lq_mgs_qr_batched_dev", dA.ptr, batch, 32, 32, 0, dQ.ptr, dR.ptr, dI.ptr)
        ctx.sync()
        Q0, R0 = np.empty_like(A), np.empty_like(A)
        ctx.call("lq_memcpy_d2h", Q0.ctypes.data, dQ.ptr, per)
        ctx.call("lq_memcpy_d2h", R0.ctypes.data, dR.ptr, per)
        ctx.sync()
        Ql, Rl = np.empty_like(A), np.empty_like(A)
        ctx.call("lq_memcpy_d2h", Ql.ctypes.data, dQ.ptr + (reps - 1) * per, per)
        ctx.call("lq_memcpy_d2h", Rl.ctypes.data, dR.ptr + (reps - 1) * per, per)
        ctx.sync()
        assert np.array_equal(Q0, Ql) and np.array_equal(R0, Rl)  # same input -> same bits, any replica
        sub = np.arange(0, uniq, 64)
        fn = orc.householder_qr_batched if which == "hh" else orc.mgs_qr_batched
        Qo, Ro = fn(A[sub])
        assert orc.rel_max_err(Q0[sub], Qo) <= REL and orc.rel_max_err(R0[sub], Ro) <= REL
        resid = np.linalg.norm(A - Q0 @ R0, axis=(1, 2)) / np.linalg.norm(A, axis=(1, 2))
        assert resid.max() <= RESID
        if which == "hh":
            G = np.swapaxes(Q0, 1, 2) @ Q0 - np.eye(32)
            assert np.abs(G).max() <= ORTH
            assert np.all(np.tril(R0, -1) == 0.0)
        else:
            info = np.empty(batch, dtype=np.int32)
            ctx.call("lq_memcpy_d2h", info.ctypes.data, dI.ptr, info.nbytes)
            ctx.sync()
            assert not info.any()


def test_mgs_dependent_columns_raise(ctx):
    A = np.random.default_rng(5).standard_normal((32, 32))
    A[:, 7] = A[:, 3]
    with pytest.raises(ValueError, match="linearly dependent"):
        lb.qr(A, ctx=ctx)
    B = np.random.default_rng(6).standard_normal((4, 32, 32))
    B[2][:, 9] = 2.0 * B[2][:, 1]
    with pytest.raises(ValueError, match="linearly dependent"):
        lb.qr_batched(B, ctx=ctx)
    with pytest.raises(ValueError, match="linearly dependent"):
        lb.qr(np.ones((6, 3)), ctx=ctx)
    with pytest.raises(ValueError):
        lb.qr(np.random.default_rng(1).standard_normal((3, 5)), ctx=ctx)  # m < n: always dependent


# ------------------------------------------------------------------ generic shapes (one CTA per matrix)
@pytest.mark.parametrize("m,n", [(1, 1), (2, 2), (7, 3), (33, 32), (64, 64), (100, 10), (128, 100), (31, 31), (200, 50)])
def test_small_generic_shapes(ctx, m, n):
    A = np.random.default_rng(1000 + m * n).standard_normal((3, m, n))
    Q, R = lb.householder_qr_batched(A, ctx=ctx)
    Qo, Ro = orc.householder_qr_batched(A)
    for i in range(3):
        check_qr(A[i], Q[i], R[i], Qo[i], Ro[i])
    Q, R = lb.qr_batched(A, ctx=ctx)
    Qo, Ro = orc.mgs_qr_batched(A)
    assert orc.rel_max_err(Q, Qo) <= REL and orc.rel_max_err(R, Ro) <= REL


# ------------------------------------------------------------------ cfg1 / cfg4: single matrix, blocked compact-WY
@pytest.mark.parametrize("m,n", [(256, 256), (300, 300), (512, 256), (700, 130), (1000, 1000), (1024, 1024), (2000, 40)])
def test_blocked_householder_vs_oracle(ctx, m, n):
    A = np.random.default_rng(m + n).standard_normal((m, n))
    Q, R = lb.householder_qr(A, ctx=ctx)
    Qo, Ro = orc.householder_qr(A)
    check_qr(A, Q, R, np.ascontiguousarray(Qo), Ro)


def test_blocked_householder_zero_columns_and_integers(ctx):
    A = np.random.default_rng(9).integers(-9, 10, (384, 200)).astype(np.float64)
    A[:, 17] = 0.0
    A[:, 130] = 0.0
    Q, R = lb.householder_qr(A, ctx=ctx)
    Qo, Ro = orc.householder_qr(A)
    check_qr(A, Q, R, np.ascontiguousarray(Qo), Ro)
    assert not np.shares_memory(Q, A)


def test_blocked_2048_lapack_crosscheck(ctx):
    """At 2048^2 the reference needs ~46 s; cross-check against LAPACK with the documented sign
    difference (last row of R / last column of Q negated, SURVEY.md 7.3-1) plus the invariants."""
    n = 2048
    A = np.random.default_rng(5).standard_normal((n, n))
    Q, R = lb.householder_qr(A, ctx=ctx)
    Ql, Rl = np.linalg.qr(A)
    Rl[-1] *= -1.0
    Ql[:, -1] *= -1.0
    assert orc.rel_max_err(R, Rl) <= REL and orc.rel_max_err(Q, Ql) <= 1e-9
    assert orc.qr_residual(A, Q, R) <= RESID and orc.orth_error(Q) <= ORTH
    assert np.all(np.tril(R, -1) == 0.0)


def test_blocked_8192_full_size_properties(ctx):
    """BASELINE cfg4 at full size, device resident.  O(n^3) checks are unaffordable on the host, so
    the invariants are probed with random vectors: A x = Q (R x), Q^T (Q x) = x, plus the sign rule
    R[j,j] = -copysign(||x||, x0) checked on column 0 and exact zeros below the diagonal."""
    n = 8192
    A = np.random.default_rng(5).standard_normal((n, n))
    dA, dQ, dR = ctx.upload(A), ctx.alloc(A.nbytes), ctx.alloc(A.nbytes)
    ctx.call("lq_householder_qr_dev", dA.ptr, n, n, dQ.ptr, dR.ptr)
    Q = ctx.download(dQ, (n, n))
    R = ctx.download(dR, (n, n))
    X = np.random.default_rng(6).standard_normal((n, 4))
    AX = A @ X
    assert np.linalg.norm(AX - Q @ (R @ X)) / np.linalg.norm(AX) <= 1e-12
    assert np.linalg.norm(Q.T @ (Q @ X) - X) / np.linalg.norm(X) <= 1e-12
    assert np.linalg.norm(Q @ (Q.T @ X) - X) / np.linalg.norm(X) <= 1e-12
    assert np.all(np.tril(R, -1) == 0.0)
    assert abs(R[0, 0] + np.copysign(np.linalg.norm(A[:, 0]), A[0, 0])) <= 1e-10 * abs(R[0, 0])
    assert np.allclose(np.abs(np.diag(R))[:8], np.abs(np.diag(np.linalg.qr(A[:, :8])[1])), rtol=1e-10)


@pytest.mark.parametrize("n", [6400, 8192])
def test_blocked_two_range_path_full_R_against_lapack(ctx, n):
    """Matrices with >= 6144 columns take the two-range trailing update / Q formation (two side streams, split at
    0.65 n).  Full R and every diagonal sign against LAPACK (np.linalg.qr, R only: ~10 s of host time at 8192^2) with
    the documented convention difference of linalg/qr.py:82-86 (the reference also reflects the last 1-element column:
    last row of R negated, SURVEY.md 7.3-1), elementwise at the north-star tolerance, plus the Q invariants on probes."""
    A = np.random.default_rng(5 + n).standard_normal((n, n))
    dA, dQ, dR = ctx.upload(A), ctx.alloc(A.nbytes), ctx.alloc(A.nbytes)
    ctx.call("lq_householder_qr_dev", dA.ptr, n, n, dQ.ptr, dR.ptr)
    R = ctx.download(dR, (n, n))
    Rl = np.linalg.qr(A, mode="r")
    Rl[-1] *= -1.0
    assert np.array_equal(np.sign(np.diag(R)), np.sign(np.diag(Rl)))          # every reflector's sign
    assert orc.rel_max_err(R, Rl) <= REL
    assert np.max(np.abs(np.diag(R) - np.diag(Rl)) / np.abs(np.diag(Rl))) <= REL
    assert np.all(np.tril(R, -1) == 0.0)
    Q = ctx.download(dQ, (n, n))
    X = np.random.default_rng(6).standard_normal((n, 4))
    AX = A @ X
    assert np.linalg.norm(AX - Q @ (R @ X)) / np.linalg.norm(AX) <= 1e-12
    assert np.linalg.norm(Q.T @ (Q @ X) - X) / np.linalg.norm(X) <= 1e-12
    for b in (dA, dQ, dR):
        b.free()


def test_gemm_building_block(ctx):
    rng = np.random.default_rng(3)
    for ta, tb, M, N, K in [(0, 0, 200, 136, 48), (1, 0, 128, 256, 4096), (0, 0, 4096, 128, 128), (1, 1, 33, 17, 9),
                            (0, 1, 130, 70, 35), (1, 0, 32, 96, 2048)]:
        Ah = rng.standard_normal((K, M) if ta else (M, K))
        Bh = rng.standard_normal((N, K) if tb else (K, N))
        Ch = rng.standard_normal((M, N))
        dA, dB, dC = ctx.upload(Ah), ctx.upload(Bh), ctx.upload(Ch)
        ctx.call("lq_gemm_dev", ta, tb, M, N, K, C.c_double(0.5), dA.ptr, Ah.shape[1], dB.ptr, Bh.shape[1],
                 C.c_double(2.0), dC.ptr, N)
        got = ctx.download(dC, (M, N))
        want = 0.5 * (Ah.T if ta else Ah) @ (Bh.T if tb else Bh) + 2.0 * Ch
        assert orc.rel_max_err(got, want) <= 1e-13, (ta, tb, M, N, K)


# ------------------------------------------------------------------ a3 / a4: least squares
@pytest.mark.parametrize("name", golden_cases("ls"))
def test_least_squares_golden(ctx, golden, name):
    A = golden[f"ls/{name}/A"]
    if name == "cfg3":
        B = golden["ls/cfg3/B"]
        X = lb.least_squares_householder_qr_batched(A, B, ctx=ctx)
        assert X.shape == (2, 64, 16) and orc.rel_max_err(X.reshape(2, -1), golden["ls/cfg3/X_hh"].reshape(2, -1)) <= REL
        X = lb.least_squares_qr_batched(A, B, ctx=ctx)
        assert X.shape == (2, 64 * 16) and orc.rel_max_err(X, golden["ls/cfg3/X_mgs"]) <= REL
        return
    b = golden[f"ls/{name}/b"]
    xh = lb.least_squares_householder_qr(A, b, ctx=ctx)
    xm = lb.least_squares_qr(A, b, ctx=ctx)
    assert xh.shape == golden[f"ls/{name}/x_hh"].shape and xm.shape == golden[f"ls/{name}/x_mgs"].shape
    if name.startswith("upper50"):
        # tests/test_qr.py:23-47: the bar is the infinity-norm residual against lstsq, rtol 1e-8
        res_np = np.linalg.norm(A @ np.linalg.lstsq(A, b, rcond=None)[0] - b, np.inf)
        bound = max(res_np * (1 + 1e-8), 1e-9 * np.linalg.norm(b, np.inf))
        assert np.linalg.norm(A @ xh - b, np.inf) <= bound
        assert np.linalg.norm(A @ xm - b, np.inf) <= bound
    else:
        assert orc.rel_max_err(xh, golden[f"ls/{name}/x_hh"]) <= REL
        assert orc.rel_max_err(xm, golden[f"ls/{name}/x_mgs"]) <= REL


def test_least_squares_cfg3_batch(ctx):
    """cfg3 shape class (256 x 64, 16 right-hand sides), 192 systems against the oracle loop."""
    A = np.random.default_rng(3).standard_normal((192, 256, 64))
    B = np.random.default_rng(4).standard_normal((192, 256, 16))
    X = lb.least_squares_householder_qr_batched(A, B, ctx=ctx)
    assert orc.rel_max_err(X, orc.lstsq_householder_batched(A, B)) <= REL
    Xm = lb.least_squares_qr_batched(A, B, ctx=ctx)
    assert orc.rel_max_err(Xm, orc.lstsq_mgs_batched(A, B)) <= REL
    # normal equations hold: A^T (A x - b) = 0
    r = A @ X - B
    g = np.swapaxes(A, 1, 2) @ r
    assert np.abs(g).max() <= 1e-10


def test_least_squares_cfg3_full_size_batch(ctx):
    """BASELINE cfg3 at its FULL batch (2^16 systems of 256 x 64 with 16 right-hand sides, device resident): 4096 distinct
    systems tiled 16 x.  The 4096-system subsample is held to LAPACK at the north-star tolerance (1e-10 per system) and to
    the normal equations A^T (A x - b) = 0; the other 15 replicas must reproduce it bit for bit (every system of the batch is
    thereby checked); same for the MGS entry point with its dependence report all clear."""
    uniq, reps, m, n, k = 4096, 16, 256, 64, 16
    A = np.random.default_rng(3).standard_normal((uniq, m, n))
    B = np.random.default_rng(4).standard_normal((uniq, m, k))
    nsys = uniq * reps
    dA, dB = ctx.alloc(8 * nsys * m * n), ctx.alloc(8 * nsys * m * k)
    for r in range(reps):
        ctx.call("lq_memcpy_h2d", dA.ptr + r * A.nbytes, A.ctypes.data, A.nbytes)
        ctx.call("lq_memcpy_h2d", dB.ptr + r * B.nbytes, B.ctypes.data, B.nbytes)
    ctx.sync()
    dX, dI = ctx.alloc(8 * nsys * n * k), ctx.alloc(4 * nsys)
    Xref = np.stack([np.linalg.lstsq(A[i], B[i], rcond=None)[0] for i in range(uniq)])
    scale = np.max(np.abs(Xref), axis=(1, 2))
    for name, extra in (("lq_lstsq_householder_batched_dev", ()), ("lq_lstsq_mgs_batched_dev", (dI.ptr,))):
        ctx.call("lq_memset", dX.ptr, 0xFF, 8 * nsys * n * k)
        ctx.call(name, dA.ptr, dB.ptr, nsys, m, n, k, dX.ptr, *extra)
        X = ctx.download(dX, (reps, uniq, n, k))
        assert np.max(np.max(np.abs(X[0] - Xref), axis=(1, 2)) / scale) <= REL, name
        g = np.swapaxes(A, 1, 2) @ (A @ X[0] - B)
        assert np.abs(g).max() <= 1e-10, name
        for r in range(1, reps):
            assert np.array_equal(X[r], X[0]), (name, r)
        if extra:
            assert not ctx.download(dI, (nsys,), dtype=np.int32).any()
    for b in (dA, dB, dX, dI):
        b.free()


@pytest.mark.parametrize("m,n,k", [(50, 50, 1), (40, 12, 3), (100, 30, 7), (300, 64, 16), (64, 64, 32), (600, 200, 5), (33, 7, 40)])
def test_least_squares_shapes(ctx, m, n, k):
    A = np.random.default_rng(m).standard_normal((m, n))
    B = np.random.default_rng(k).standard_normal((m, k))
    x = lb.least_squares_householder_qr(A, B, ctx=ctx)
    assert x.shape == (n, k) and orc.rel_max_err(x, orc.lstsq_householder(A, B)) <= 1e-9
    xm = lb.least_squares_qr(A, B, ctx=ctx)
    assert xm.shape == (n * k,) and orc.rel_max_err(xm, orc.lstsq_mgs(A, B)) <= 1e-9
    xv = lb.least_squares_householder_qr(A, B[:, 0], ctx=ctx)
    assert xv.shape == (n,) and orc.rel_max_err(xv, x[:, 0]) <= 1e-12


# ------------------------------------------------------------------ a5: svd via A^T A
def _align(Vt, Vt_ref):
    return np.sign(np.sum(Vt * Vt_ref, axis=1))


@pytest.mark.parametrize("name", golden_cases("svd"))
def test_svd_golden(ctx, golden, name):
    A = golden[f"svd/{name}/A"]
    np.random.seed(999)
    U, s, Vt = lb.svd(A, ctx=ctx)
    s_ref, Vt_ref = golden[f"svd/{name}/s"], golden[f"svd/{name}/Vt"]
    assert s.shape == s_ref.shape and Vt.shape == Vt_ref.shape
    np.testing.assert_allclose(s, s_ref, rtol=1e-10, atol=1e-12)  # tests/test_svd.py:52
    r = int(np.sum(s_ref > 1e-8))
    sg = _align(Vt[:r], Vt_ref[:r])
    assert orc.rel_max_err(Vt[:r] * sg[:, None], Vt_ref[:r]) <= 1e-8  # tests/test_svd.py:56-57
    k = min(A.shape)
    assert np.linalg.norm((U[:, :k] * s[:k]) @ Vt[:k] - A) < 1e-10  # tests/test_svd.py:24
    if A.shape[0] >= A.shape[1]:
        assert np.abs(U.T @ U - np.eye(U.shape[1])).max() <= 1e-10  # also the completed columns
    assert np.abs(Vt @ Vt.T - np.eye(Vt.shape[0])).max() <= 1e-10
    if f"svd/{name}/U" in golden:
        U_ref = golden[f"svd/{name}/U"]
        assert U.shape == U_ref.shape
        if A.shape[0] >= A.shape[1]:
            assert orc.rel_max_err(U[:, :r] * sg[None, :r], U_ref[:, :r]) <= 1e-8


def test_svd_tall_skinny(ctx):
    A = np.random.default_rng(6).standard_normal((1 << 17, 128))
    U, s, Vt = lb.svd(A, ctx=ctx)
    _, so, Vto = orc.svd_gram(A)
    assert np.max(np.abs(s - so) / so) <= REL
    assert np.linalg.norm((U * s) @ Vt - A) / np.linalg.norm(A) <= 1e-12
    assert np.abs(U.T @ U - np.eye(128)).max() <= 1e-10
    assert np.all(np.diff(s) <= 0)


def test_svd_more_than_256_columns(ctx):
    A = np.random.default_rng(77).standard_normal((1500, 300))
    U, s, Vt = lb.svd(A, ctx=ctx)
    assert np.max(np.abs(s - np.linalg.svd(A, compute_uv=False)) / s) <= REL
    assert np.abs(U.T @ U - np.eye(300)).max() <= 1e-10 and np.abs(Vt @ Vt.T - np.eye(300)).max() <= 1e-10
    assert np.linalg.norm((U * s) @ Vt - A) / np.linalg.norm(A) <= 1e-12


def test_eigh_building_block(ctx):
    for n in (1, 2, 5, 64, 127, 128, 200, 258, 400):  # > 256: more rotations per round than threads in the replay
        M = np.random.default_rng(n).standard_normal((n + 5, n))
        G = M.T @ M
        dG, dl, dV = ctx.upload(G), ctx.alloc(8 * n), ctx.alloc(8 * n * n)
        ctx.call("lq_eigh_dev", dG.ptr, n, dl.ptr, dV.ptr)
        lam = ctx.download(dl, (n,))
        V = ctx.download(dV, (n, n))
        ref = np.linalg.eigvalsh(G)[::-1]
        assert np.max(np.abs(lam - ref)) <= 1e-12 * ref[0]
        assert np.abs(V.T @ V - np.eye(n)).max() <= 1e-12
        assert np.abs(G @ V - V * lam).max() <= 1e-11 * ref[0]


# ------------------------------------------------------------------ a7: TSQR
def test_tsqr_matches_mgs_convention(ctx, golden):
    A = golden["tsqr/mgs_1024x64/A"]
    Q, R = lb.tsqr(A, ctx=ctx)
    assert orc.rel_max_err(R, golden["tsqr/mgs_1024x64/R"]) <= REL
    assert np.all(np.diag(R) > 0) and np.all(np.tril(R, -1) == 0.0)
    assert orc.qr_residual(A, Q, R) <= RESID and orc.orth_error(Q) <= ORTH
    Qm, Rm = orc.mgs_qr(A)
    assert orc.rel_max_err(Q, Qm) <= 1e-9


@pytest.mark.parametrize("m,n", [(128, 128), (1000, 17), (5000, 100), (1 << 16, 128), (300001, 64)])
def test_tsqr_shapes(ctx, m, n):
    A = np.random.default_rng(m % 1000 + n).standard_normal((m, n))
    Q, R = lb.tsqr(A, ctx=ctx)
    Qo, Ro = orc.tsqr_reference(A)
    assert orc.rel_max_err(R, Ro) <= REL and orc.rel_max_err(Q, Qo) <= 1e-9
    assert orc.qr_residual(A, Q, R) <= RESID and orc.orth_error(Q) <= ORTH


def test_tsqr_ill_conditioned_falls_back_to_householder(ctx):
    """cond(A) ~ 1e9+: the CholeskyQR2 fast path must hand over to the reflector-based path and stay O(eps)."""
    A = np.random.default_rng(3).standard_normal((20000, 32)) * np.logspace(0, -9, 32)
    A[:, 5] = A[:, 4] * (1 + 1e-9) + 1e-9 * A[:, 6]
    Q, R = lb.tsqr(A, ctx=ctx)
    assert np.all(np.diag(R) > 0) and np.all(np.tril(R, -1) == 0.0)
    assert orc.qr_residual(A, Q, R) <= RESID and orc.orth_error(Q) <= ORTH


# ------------------------------------------------------------------ section 8(f) "next" rows: callers of the path
def test_project_onto_colspace(ctx):
    # the reference's hand-computed case, tests/test_projections.py:12-44
    A = np.array([[1, 0], [1, 1], [1, 2]])
    b = np.array([[6], [0], [0]])
    p = lb.project_onto_colspace(A, b, ctx=ctx)
    np.testing.assert_allclose(p, np.array([[5], [2], [-1]]), atol=1e-12)
    res = np.linalg.norm(A @ np.linalg.lstsq(A, b, rcond=None)[0] - b, np.inf)
    assert abs(res - np.linalg.norm(p - b, np.inf)) < 1e-12
    # random tall matrix, several right-hand sides, and a rank-deficient one (pseudo-inverse branch upstream)
    rng = np.random.default_rng(8)
    A = rng.standard_normal((300, 40)); B = rng.standard_normal((300, 5))
    P = lb.project_onto_colspace(A, B, ctx=ctx)
    assert orc.rel_max_err(P, A @ np.linalg.lstsq(A, B, rcond=None)[0]) <= 1e-10
    A[:, 7] = A[:, 3] + A[:, 4]
    P = lb.project_onto_colspace(A, B[:, 0], ctx=ctx)
    assert P.shape == (300, 1)
    assert orc.rel_max_err(P, A @ (np.linalg.pinv(A) @ B[:, :1])) <= 1e-9


def test_pca_matches_numpy(ctx):
    rng = np.random.default_rng(21)
    A = rng.standard_normal((500, 12)) @ np.diag(np.linspace(3.0, 0.5, 12)) + 4.0
    k = 5
    pcs, scores, ev, evr, tv, mean_ = lb.pca(A, k, ctx=ctx)
    X = A - A.mean(axis=0)
    _, S, Vt = np.linalg.svd(X, full_matrices=False)
    np.testing.assert_allclose(ev, S[:k] ** 2 / 499, rtol=1e-10)
    np.testing.assert_allclose(tv, np.linalg.norm(X) ** 2 / 499, rtol=1e-12)
    np.testing.assert_allclose(evr, ev / tv, rtol=1e-12)
    np.testing.assert_allclose(mean_, A.mean(axis=0), rtol=1e-14)
    sg = np.sign(np.sum(pcs * Vt[:k].T, axis=0))
    assert orc.rel_max_err(pcs * sg, Vt[:k].T) <= 1e-8
    assert orc.rel_max_err(scores * sg, X @ Vt[:k].T) <= 1e-8
    assert np.abs(pcs.T @ pcs - np.eye(k)).max() <= 1e-10


# ------------------------------------------------------------------ batched 32 x 32 Householder kernel
@pytest.mark.parametrize("batch", [1, 5, 31, 33, 1000, 4099])
def test_batched32_householder_kernel_matches_oracle(ctx, batch):
    """The 32 x 32 kernel of a1 (lane = column, left-looking panels, Q formed by compact-WY block reflectors on
    DMMA.8x8x4) against the reference semantics (oracle, 1e-10) and the QR invariants over the whole batch, with ragged
    tails, a skipped reflector (qr.py:79: zero column), a dependent column and a badly scaled matrix.  It is the only
    kernel variant: any other variant number is an argument error."""
    rng = np.random.default_rng(900 + batch)
    A = rng.standard_normal((batch, 32, 32))
    if batch > 16:
        A[3, :, 5] = 0.0            # skipped reflector
        A[7, :, 9] = A[7, :, 2]     # dependent column
        A[11] *= 1e-9               # small scale (absolute 1e-12 threshold not reached)
        A[12] *= 1e7
        A[13, :, 0] = 0.0           # first column skipped
        A[14, :, 31] = 0.0          # last column skipped
    dA = ctx.upload(A)
    dQ, dR = ctx.upload(np.full_like(A, np.nan)), ctx.upload(np.full_like(A, np.nan))
    with pytest.raises(ValueError, match="variant 14 does not exist"):
        ctx.call("lq_householder_qr_batched_dev", dA.ptr, batch, 32, 32, dQ.ptr, dR.ptr, 14)
    ctx.call("lq_householder_qr_batched_dev", dA.ptr, batch, 32, 32, dQ.ptr, dR.ptr, 0)
    Qv, Rv = ctx.download(dQ, A.shape), ctx.download(dR, A.shape)
    assert np.isfinite(Qv).all() and np.isfinite(Rv).all()
    assert np.all(np.tril(Rv, -1) == 0.0)
    nref = min(batch, 48)
    Qo, Ro = orc.householder_qr_batched(A[:nref])
    for i in range(nref):
        if batch > 16 and i == 7:
            # dependent column: the reflector of column 9 is built from rounding noise, Q is not unique there;
            # the invariants still hold
            assert orc.qr_residual(A[i], Qv[i], Rv[i]) <= 1e-12 and orc.orth_error(Qv[i]) <= 1e-12, i
            continue
        assert orc.rel_max_err(Qv[i], Qo[i]) <= REL and orc.rel_max_err(Rv[i], Ro[i]) <= REL, i
    # every matrix of the batch: invariants
    resid = np.linalg.norm(A - Qv @ Rv, axis=(1, 2)) / np.linalg.norm(A, axis=(1, 2))
    orth = np.abs(np.swapaxes(Qv, 1, 2) @ Qv - np.eye(32)).max(axis=(1, 2))
    assert resid.max() <= 1e-12 and orth.max() <= 1e-12, (resid.max(), orth.max())


@pytest.mark.parametrize("m", [33, 64, 300, 1000, 4096, 8192])
def test_panel_kernel_versions_agree(ctx, m):
    """The panel factorisations of the blocked path (barrier.cluster kernel, st.async kernel with 256 rows per CTA, and
    the default choice, which is the one-CTA SOLO kernel up to 256 rows) produce the same R rows, unit-norm reflectors
    and compact-WY factor, and (I - V T V^T)^T A = [R; 0].  Versions 2 and 4 do not exist."""
    lda = 64
    A = np.random.default_rng(m).standard_normal((m, 32))
    if m == 300:
        A[:, 7] = 0.0
        A[:, 20] = A[:, 3]

    def run(version):
        buf = np.zeros((m, lda))
        buf[:, :32] = A
        dA, dV, dT = ctx.upload(buf), ctx.upload(np.zeros((m, lda))), ctx.upload(np.zeros((32, 128)))
        ctx.call("lq_debug_panel", dA.ptr, lda, dV.ptr, lda, dT.ptr, 128, m, 32, version)
        R = np.triu(ctx.download(dA, (m, lda))[:32, :32])
        return R, ctx.download(dV, (m, lda))[:, :32].copy(), ctx.download(dT, (32, 128))[:, :32].copy()

    ref = run(1)
    scale = np.abs(A).max()
    for version in (3, 0):
        if version == 3 and m > 16 * 256:
            continue
        R, V, T = run(version)
        assert orc.rel_max_err(R, ref[0]) <= 1e-13 and orc.rel_max_err(V, ref[1]) <= 1e-13 and orc.rel_max_err(T, ref[2]) <= 1e-12
        QtA = A - V @ (T.T @ (V.T @ A))
        assert np.abs(QtA[:32] - R).max() <= 1e-13 * scale * np.sqrt(m) and (m == 32 or np.abs(QtA[32:]).max() <= 1e-13 * scale * np.sqrt(m))
    for version in (2, 4):
        with pytest.raises(ValueError):
            run(version)


def test_eigh_one_sided_matches_two_sided(ctx):
    """n <= 128 runs the one-sided block round-robin Jacobi; the JACOBI_TWO_SIDED option selects the two-sided kernel."""
    for n, rows in ((128, 4096), (128, 100), (96, 500), (33, 40)):
        M = np.random.default_rng(n + rows).standard_normal((rows, n))
        G = M.T @ M
        res = {}
        for two in (False, True):
            ctx.set_option("JACOBI_TWO_SIDED", two)
            try:
                dG, dl, dV = ctx.upload(G), ctx.alloc(8 * n), ctx.alloc(8 * n * n)
                ctx.call("lq_eigh_dev", dG.ptr, n, dl.ptr, dV.ptr)
                res[two] = (ctx.download(dl, (n,)), ctx.download(dV, (n, n)))
            finally:
                ctx.set_option("JACOBI_TWO_SIDED", False)
        ref = np.linalg.eigvalsh(G)[::-1]
        for lam, V in res.values():
            assert np.max(np.abs(lam - ref)) <= 1e-12 * ref[0]
            assert np.abs(V.T @ V - np.eye(n)).max() <= 1e-12
            assert np.abs(G @ V - V * lam).max() <= 1e-11 * ref[0]
        assert np.max(np.abs(res[False][0] - res[True][0])) <= 1e-12 * ref[0]


def test_no_cpu_fallback_loaded(ctx):
    """The numbers above came from the in-tree CUDA library: it is the loaded object and it counted launches."""
    from linalg_b200 import _native

    assert ctx.launches() > 0
    maps = open("/proc/self/maps").read()
    assert _native.LIB_PATH in maps


# ----------------------------------------------------------------------------- section 8(f): remaining rows
def test_adjugate_matches_reference_contract(ctx):
    """tests/test_matrix_functions.py:21-28 (adj vs det * inv, atol 1e-8) for the one-matrix and the batched form, plus the
    singular branch of linalg/matrix_functions.py:48-58 (cofactors) on an exactly singular matrix."""
    rng = np.random.default_rng(21)
    A = rng.standard_normal((10, 10))
    assert np.allclose(lb.adj(A, ctx=ctx), np.linalg.det(A) * np.linalg.inv(A), atol=1e-8)
    assert np.isclose(lb.det(A, ctx=ctx), np.linalg.det(A), rtol=1e-10)
    Ab = rng.standard_normal((257, 12, 12))
    ref = np.linalg.det(Ab)[:, None, None] * np.linalg.inv(Ab)
    got = lb.adj_batched(Ab, ctx=ctx)
    assert np.max(np.abs(got - ref) / np.max(np.abs(ref), axis=(1, 2), keepdims=True)) <= 1e-10
    assert np.allclose(lb.det_batched(Ab, ctx=ctx), np.linalg.det(Ab), rtol=1e-10)
    S = np.array([[1.0, 2.0, 3.0], [0.0, 0.0, 0.0], [4.0, 5.0, 6.0]])          # det == 0 exactly: cofactor branch
    assert lb.det(S, ctx=ctx) == 0.0
    cof = np.array([[0.0, 3.0, 0.0], [0.0, -6.0, 0.0], [0.0, 3.0, 0.0]])          # hand-computed adjugate
    assert np.allclose(lb.adj(S, ctx=ctx), cof, atol=1e-12)
    with pytest.raises(ValueError):
        lb.adj(np.ones((3, 4)), ctx=ctx)


def test_random_nonsingular_qr_batched(ctx):
    """linalg/qr.py:137-154 for a list of seeds in one batched MGS call: every matrix equals the one-matrix drop-in bitwise
    and the reference's algorithm (oracle MGS on the same default_rng draws) to rounding; columns orthogonal with the drawn
    norms, i.e. non-singular -- what tests/test_elimination.py:71-103 relies on."""
    seeds = [0, 1, 7, 123, 2 ** 31]
    M = lb.random_nonsingular_qr_batched(9, seeds, ctx=ctx)
    for i, sd in enumerate(seeds):
        assert np.array_equal(M[i], lb.random_nonsingular_qr(9, seed=sd, ctx=ctx))
        rng = np.random.default_rng(sd)
        A0 = rng.standard_normal((9, 9))
        Qo, _ = orc.mgs_qr(A0)
        sc = rng.uniform(0.5, 10.0, size=9)
        assert orc.rel_max_err(M[i], Qo * sc) <= 1e-10
        G = M[i].T @ M[i]
        assert np.allclose(G, np.diag(sc ** 2), atol=1e-10)


def test_svd_rank_deficient_device_seeded(ctx):
    """seed= (SURVEY.md 8f-1): the completion of linalg/svd.py:67-76 from device-generated candidates -- deterministic,
    and the invariants tests/test_svd.py:60-79 pins hold; seed=None keeps the upstream (global np.random) behaviour."""
    for k in (1, 3):
        A = np.random.default_rng(123 + k).normal(size=(10, 7))
        A[:, -k:] = 0.0
        U1, s1, Vt1 = lb.svd(A, ctx=ctx, seed=42)
        U2, s2, Vt2 = lb.svd(A, ctx=ctx, seed=42)
        assert np.array_equal(U1, U2) and np.array_equal(s1, s2)
        U3, _, _ = lb.svd(A, ctx=ctx, seed=43)
        assert not np.array_equal(U1[:, -k:], U3[:, -k:])
        r = 7 - k
        assert np.all(s1[:r] > 1e-12) and np.all(s1[r:] < 1e-12)
        assert np.linalg.norm((U1 * s1) @ Vt1 - A) < 1e-10
        assert np.allclose(U1.T @ U1, np.eye(7), atol=1e-10)
    # the generator itself: N(0, 1) moments, a function of (seed, index) only
    n = 1 << 20
    d1, d2 = ctx.alloc(8 * n), ctx.alloc(8 * (n // 2 + 3))
    ctx.call("lq_random_normal_dev", d1.ptr, n, 5)
    ctx.call("lq_random_normal_dev", d2.ptr, n // 2 + 3, 5)
    z, z2 = ctx.download(d1, (n,)), ctx.download(d2, (n // 2 + 3,))
    assert np.array_equal(z[: n // 2 + 3], z2)
    assert abs(z.mean()) < 5e-3 and abs(z.std() - 1.0) < 5e-3 and abs(np.mean(z ** 4) - 3.0) < 5e-2
    assert np.all(np.isfinite(z)) and len(np.unique(z)) > 0.999 * n


def test_least_squares_householder_singular_raises_like_numpy(ctx):
    """A zero column leaves R[j, j] exactly 0; the reference's np.linalg.solve(R, Q^T b) (linalg/qr.py:134) raises
    LinAlgError("Singular matrix") there -- so do the drop-in entry points (ADVICE r1), one-matrix and batched."""
    rng = np.random.default_rng(31)
    A = rng.standard_normal((40, 6))
    A[:, 2] = 0.0
    b = rng.standard_normal(40)
    with pytest.raises(np.linalg.LinAlgError):
        orc.lstsq_householder(A, b)
    with pytest.raises(np.linalg.LinAlgError):
        lb.least_squares_householder_qr(A, b, ctx=ctx)
    Ab = rng.standard_normal((9, 256, 64))
    Bb = rng.standard_normal((9, 256, 16))
    X = lb.least_squares_householder_qr_batched(Ab, Bb, ctx=ctx)          # regular batch: no report
    assert orc.rel_max_err(X, orc.lstsq_householder_batched(Ab, Bb)) <= REL
    Ab[7, :, 63] = 0.0
    with pytest.raises(np.linalg.LinAlgError):
        lb.least_squares_householder_qr_batched(Ab, Bb, ctx=ctx)


def test_blocked_graph_replay_is_bitwise_identical(ctx):
    """lq_householder_qr_dev replays the blocked multi-stream schedule as a CUDA graph from the third call with the same
    shape and buffers (first call: plain launches, second: capture).  Every call must return the same bits, also after the
    input buffer's CONTENT changes (the graph holds pointers, not data), and LINALG_B200_NO_GRAPH-style plain launches on
    other buffers must agree."""
    n = 320
    rng = np.random.default_rng(91)
    A1, A2 = rng.standard_normal((n, n)), rng.standard_normal((n, n))
    dA, dQ, dR = ctx.upload(A1), ctx.alloc(A1.nbytes), ctx.alloc(A1.nbytes)
    outs = []
    for it in range(4):
        ctx.call("lq_householder_qr_dev", dA.ptr, n, n, dQ.ptr, dR.ptr)
        outs.append((ctx.download(dQ, (n, n)), ctx.download(dR, (n, n))))
    for Q, R in outs[1:]:
        assert np.array_equal(Q, outs[0][0]) and np.array_equal(R, outs[0][1])
    Qo, Ro = orc.householder_qr(A1)
    assert orc.rel_max_err(outs[-1][0], Qo) <= REL and orc.rel_max_err(outs[-1][1], Ro) <= REL
    ctx.upload(A2, dA)                                        # same buffers, new matrix: the replayed graph must factor A2
    ctx.call("lq_householder_qr_dev", dA.ptr, n, n, dQ.ptr, dR.ptr)
    Q2, R2 = ctx.download(dQ, (n, n)), ctx.download(dR, (n, n))
    dB, dQ2, dR2 = ctx.upload(A2), ctx.alloc(A2.nbytes), ctx.alloc(A2.nbytes)
    ctx.call("lq_householder_qr_dev", dB.ptr, n, n, dQ2.ptr, dR2.ptr)   # other buffers: first call = plain launches
    assert np.array_equal(Q2, ctx.download(dQ2, (n, n))) and np.array_equal(R2, ctx.download(dR2, (n, n)))
    assert orc.qr_residual(A2, Q2, R2) <= RESID and orc.orth_error(Q2) <= ORTH
    for b in (dA, dQ, dR, dB, dQ2, dR2):
        b.free()


def test_svd_direct_eigenvectors_and_replay_agree(ctx):
    """For a well-conditioned Gram matrix (lambda_min > 1e-2 lambda_max) svd takes the eigenvectors as the normalised converged
    Jacobi columns instead of replaying the rotation log; a matrix just outside that window replays.  Both must satisfy the
    reference's contract (tests/test_svd.py:13-57: s vs LAPACK 1e-10, orthogonality, reconstruction) at the north-star
    tolerances, for full n = 128 and a padded n."""
    rng = np.random.default_rng(77)
    for n, spread in ((128, 1.0), (128, 30.0), (100, 2.0), (37, 1.0)):
        A = rng.standard_normal((6000, n)) * np.linspace(1.0, spread, n)[None, :]
        U, s, Vt = lb.svd(A, ctx=ctx)
        so = np.linalg.svd(A, compute_uv=False)
        assert np.max(np.abs(s - so) / so) <= 1e-10, (n, spread)
        assert np.abs(U.T @ U - np.eye(n)).max() <= 1e-12 and np.abs(Vt @ Vt.T - np.eye(n)).max() <= 1e-12, (n, spread)
        assert np.linalg.norm((U * s) @ Vt - A) / np.linalg.norm(A) <= 1e-12, (n, spread)

"""Every kernel route of the QR and least-squares entry points, at the shapes where the choice of route changes.

Kernel selection depends on the shape alone: each entry point is a fixed table of routes picked by thresholds on
(m, n, nrhs) and on the device's opt-in shared memory per block.  The functions below mirror those predicates
(``batched_small.cuh``, ``lstsq_stream.cu``, ``lq_householder_qr_dev`` in ``blocked_qr.cu``, ``stage_host`` in
``api_host.cu``) and derive the boundary shapes from them, so a case sits on the last shape of a route or on the
first shape of the next one.  Every call also counts kernel launches: a one-kernel route launches exactly once per call
(once per chunk on the host pipelines), a blocked or large route more than once per matrix.  A mirror that drifts from
the library fails there, instead of quietly turning a boundary case into a duplicate of its neighbour.

References: Q and R against the oracle (the reference's algorithm and sign convention) at the 1e-10 bar; X against
Householder QR carried out in extended precision, to the normwise bound 4 max(m, n) u kappa (1 + kappa eta) (kappa^2 for
the MGS routes), which LAPACK's solution has to meet on the same input as well.
"""
import functools

import numpy as np
import pytest

import linalg_b200 as lb
from linalg_b200 import _native
from oracle import linalg_oracle as orc

pytestmark = pytest.mark.gpu

REL = 1e-10
RESID = 1e-12
ORTH = 1e-12
U64 = 2.0 ** -53


# ----------------------------------------------------------------------------- the route table
def small_pitch(m):
    return m if m & 1 else m + 1


def small_hh_smem_doubles(m, n, nrhs):
    return small_pitch(m) * (n + nrhs) + 3 * n + 64


def small_mgs_smem_doubles(m, n, nrhs):
    return small_pitch(m) * (n + nrhs) + n * (n + nrhs) + 64


def tile_fits(m, n, nrhs):  # lstsq_tile_kernel: one warp per system
    return 1 <= n <= 64 and 1 <= nrhs <= 16 and m >= n


def stream_fits(m, n, nrhs):  # lstsq_stream_kernel: 64-row blocks; Householder entry points only
    return 1 <= n <= 64 and 1 <= nrhs <= 32 and m >= n


SINGLE_SMALL_MN = 4096      # lq_householder_qr_dev keeps m * n <= 4096 on the one-CTA kernel
CHUNK_BYTES = 192 << 20     # host pipelines: about 192 MiB of device traffic per chunk


def chunk_of(bytes_per_item):
    return max(1, CHUNK_BYTES // bytes_per_item)


def hh_qr_route(m, n, smem, batched):
    if batched and m == n == 32:
        return "qr32"
    if not batched and m * n > SINGLE_SMALL_MN:
        return "blocked"
    return "small" if 8 * small_hh_smem_doubles(m, n, 0) <= smem else "blocked"


def mgs_qr_route(m, n, smem):
    if m == n == 32:
        return "qr32"
    return "small" if 8 * small_mgs_smem_doubles(m, n, 0) <= smem else "large"


def lstsq_route(method, m, n, nrhs, smem):
    if tile_fits(m, n, nrhs):
        return "tile"
    if method == "hh" and stream_fits(m, n, nrhs):
        return "stream"
    need = small_hh_smem_doubles if method == "hh" else small_mgs_smem_doubles
    return "small" if 8 * need(m, n, nrhs) <= smem else "large"


ONE_KERNEL = {"qr32", "small", "tile", "stream"}


def last_fitting(fits):
    """Largest x >= 1 with fits(x), for a predicate that holds at 1 and fails from some x on."""
    assert fits(1)
    lo, hi = 1, 2
    while fits(hi):
        lo, hi = hi, 2 * hi
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (mid, hi) if fits(mid) else (lo, mid)
    return lo


def boundary(name, smem):
    """(last shape of the one-CTA route, first shape of the next route) for the named family."""
    hh = lambda m, n, k: 8 * small_hh_smem_doubles(m, n, k) <= smem
    mgs = lambda m, n, k: 8 * small_mgs_smem_doubles(m, n, k) <= smem
    if name == "hh_square":
        n = last_fitting(lambda x: hh(x, x, 0))
        return (n, n), (n + 1, n + 1)
    if name == "hh_tall2":
        m = last_fitting(lambda x: hh(x, 2, 0))
        return (m, 2), (m + 1, 2)
    if name == "mgs_square":
        n = last_fitting(lambda x: mgs(x, x, 0))
        return (n, n), (n + 1, n + 1)
    if name == "mgs_tall2":
        m = last_fitting(lambda x: mgs(x, 2, 0))
        return (m, 2), (m + 1, 2)
    if name == "hh_ls":   # one-CTA least squares, 65 columns (beyond the stream kernel), one right-hand side
        m = last_fitting(lambda x: hh(max(x, 65), 65, 1))
        return (m, 65, 1), (m + 1, 65, 1)
    if name == "mgs_ls":
        m = last_fitting(lambda x: mgs(max(x, 65), 65, 1))
        return (m, 65, 1), (m + 1, 65, 1)
    raise KeyError(name)


@pytest.fixture(scope="module")
def smem(ctx):
    return ctx.props()["max_smem"]


def counted(ctx, fn, /, *args, **kw):
    """fn(*args, **kw) and the number of kernels it launched on ctx (kw may hold ctx= for fn itself)."""
    l0 = ctx.launches()
    out = fn(*args, **kw)
    return out, ctx.launches() - l0


def assert_route(route, launches, matrices, chunks=1):
    """A one-kernel route launches once per chunk; a blocked / large route more than once per matrix."""
    if route in ONE_KERNEL:
        assert launches == chunks, (route, launches, chunks)
    else:
        assert launches > matrices, (route, launches, matrices)


def test_route_table_boundaries_on_this_device(smem):
    """The derived boundaries straddle a route change (on a 227 KB device: 168 / 169, 120 / 121)."""
    for name, route_of in (("hh_square", lambda s: hh_qr_route(*s, smem, True)),
                           ("hh_tall2", lambda s: hh_qr_route(*s, smem, True)),
                           ("mgs_square", lambda s: mgs_qr_route(*s, smem)),
                           ("mgs_tall2", lambda s: mgs_qr_route(*s, smem)),
                           ("hh_ls", lambda s: lstsq_route("hh", *s, smem)),
                           ("mgs_ls", lambda s: lstsq_route("mgs", *s, smem))):
        last, first = boundary(name, smem)
        assert route_of(last) == "small" and route_of(first) in ("blocked", "large"), (name, last, first)
    if smem == 232448:
        assert boundary("hh_square", smem) == ((168, 168), (169, 169))
        assert boundary("mgs_square", smem) == ((120, 120), (121, 121))


# ----------------------------------------------------------------------------- references
if np.finfo(np.longdouble).nmant >= 63:
    def _hp(a):
        return np.array(a, dtype=np.longdouble)

    _hp_sqrt = np.sqrt
else:  # long double is plain double on this platform: 40 significant digits through mpmath instead
    import mpmath

    mpmath.mp.dps = 40

    def _hp(a):
        return np.vectorize(mpmath.mpf, otypes=[object])(np.asarray(a, dtype=np.float64))

    _hp_sqrt = mpmath.sqrt


def hp_householder(A, B=None, want_q=False, eps=orc.EPS):
    """Householder QR of A (m >= n) in extended precision with the reference's conventions (linalg/qr.py:75-97):
    R[j, j] = -copysign(||x||, x[0]), a column with ||x|| < eps (the reference's 1e-12) or ||x|| == 0 is skipped.  Returns
    (Q or None, R, X), X = R^-1 (Q^T B) for a B, else None; rounded to float64."""
    m, n = A.shape
    W = _hp(A if B is None else np.hstack([A, B]))
    refl = [None] * n
    for j in range(n):
        x = W[j:, j]
        nx = _hp_sqrt(np.sum(x * x))
        if nx < eps or nx == 0:
            continue
        v = x.copy()
        v[0] += -nx if np.signbit(np.float64(x[0])) else nx
        beta = 2 / np.sum(v * v)
        W[j:, j:] -= np.outer(v * beta, v @ W[j:, j:])
        refl[j] = (v, beta)
    R = np.triu(W[:n, :n])
    X = None
    if B is not None:
        Y = W[:n, n:].copy()
        for i in range(n - 1, -1, -1):
            if i + 1 < n:
                Y[i] -= R[i, i + 1:] @ Y[i + 1:]
            Y[i] /= R[i, i]
        X = Y.astype(np.float64)
    Q = None
    if want_q:
        Qw = _hp(np.eye(m, n))
        for j in range(n - 1, -1, -1):
            if refl[j] is not None:
                v, beta = refl[j]
                Qw[j:, j:] -= np.outer(v * beta, v @ Qw[j:, j:])
        Q = Qw.astype(np.float64)
    return Q, R.astype(np.float64), X


def ref_householder_qr(A):
    """The oracle where its full max(m, n)-square Q is affordable, the same algorithm in extended precision beyond."""
    if A.shape[0] <= 2048:
        Q, R = orc.householder_qr(A)
        return np.ascontiguousarray(Q), R
    Q, R, _ = hp_householder(A, want_q=True)
    return Q, R


def conditioned(rng, m, n, kappa):
    """U diag(s) V^T with singular values spread geometrically from 1 to 1 / kappa."""
    Um, _ = np.linalg.qr(rng.standard_normal((m, n)))
    V, _ = np.linalg.qr(rng.standard_normal((n, n)))
    return (Um * np.logspace(0, -np.log10(kappa), n)) @ V.T


@functools.lru_cache(maxsize=None)
def ls_systems(m, n, k):
    """Six systems of one shape and their extended-precision solutions: random normal; kappa 1e2 and 1e6 with
    b = A x* + a small residual; kappa 1e6 with a random b; the random one scaled by 1e-9 and by 1e7."""
    rng = np.random.default_rng(1_000_003 * m + 1009 * n + k)
    A0 = rng.standard_normal((m, n))
    A, B = [A0], [rng.standard_normal((m, k))]
    for kappa in (1e2, 1e6):
        Ak = conditioned(rng, m, n, kappa)
        AX = Ak @ rng.standard_normal((n, k))
        A.append(Ak)
        B.append(AX + 1e-10 * np.linalg.norm(AX) / np.sqrt(m * k) * rng.standard_normal((m, k)))
    A.append(conditioned(rng, m, n, 1e6))
    B.append(rng.standard_normal((m, k)))
    A += [1e-9 * A0, 1e7 * A0]
    B += [B[0], B[0]]
    A, B = np.stack(A), np.stack(B)
    Xhp = np.stack([hp_householder(A[s], B[s])[2] for s in range(len(A))])
    return A, B, Xhp


def check_x(X, A, B, Xhp, method):
    """Per right-hand side: ||x - x_hp|| / ||x_hp|| <= 4 max(m, n) u kappa (1 + kappa eta), eta = ||r|| / (||A|| ||x||)
    (MGS: 4 max(m, n) u kappa^2 (1 + eta)); LAPACK's solution meets the same bound."""
    m, n = A.shape
    s = np.linalg.svd(A, compute_uv=False)
    kappa = s[0] / s[-1]
    Xl = np.linalg.lstsq(A, B, rcond=None)[0]
    assert np.isfinite(X).all()
    for c in range(B.shape[1]):
        x = Xhp[:, c]
        nx = np.linalg.norm(x)
        eta = np.linalg.norm(B[:, c] - A @ x) / (s[0] * nx)
        if method == "hh":
            bound = 4 * max(m, n) * U64 * kappa * (1 + kappa * eta)
        else:
            bound = 4 * max(m, n) * U64 * kappa ** 2 * (1 + eta)
        assert np.linalg.norm(Xl[:, c] - x) / nx <= bound, ("lapack", c, kappa, eta)
        assert np.linalg.norm(X[:, c] - x) / nx <= bound, (c, kappa, eta, np.linalg.norm(X[:, c] - x) / nx, bound)


# ----------------------------------------------------------------------------- edge matrices
def edge_variants(A):
    """(label, matrix): the input, zero first / middle / last columns (skipped reflectors), an exactly dependent column,
    and the input scaled by 1e-9 and 1e7."""
    m, n = A.shape
    out = [("normal", A)]
    for j in sorted({0, n // 2, n - 1}):
        Z = A.copy()
        Z[:, j] = 0.0
        out.append((f"zero{j}", Z))
    if n >= 2:
        D = A.copy()
        D[:, n // 2] = 2.0 * D[:, 0]
        out.append(("dependent", D))
    out += [("scale1e-9", 1e-9 * A), ("scale1e7", 1e7 * A)]
    return out


def check_householder(label, A, Q, R, Qo=None, Ro=None):
    assert np.all(np.tril(R, -1) == 0.0), label
    assert orc.qr_residual(A, Q, R) <= RESID and orc.orth_error(Q) <= ORTH, label
    if label != "dependent":  # a reflector built from rounding noise: Q is not unique there, the invariants hold
        if Qo is None:
            Qo, Ro = ref_householder_qr(A)
        assert orc.rel_max_err(Q, Qo) <= REL and orc.rel_max_err(R, Ro) <= REL, label


# ----------------------------------------------------------------------------- Householder QR
@pytest.mark.parametrize("m,n", [(64, 64), (4096, 1), (65, 64), (100, 80), (130, 129), (255, 200), (5000, 1)])
def test_householder_qr_single_matrix_routes(ctx, smem, m, n):
    """The one-matrix entry point: m * n <= 4096 on the one-CTA kernel, beyond on the blocked path, which here runs with
    m < 256 (scratch separate from the A workspace), with n = 1 and with n % 32 != 0 (padded columns)."""
    route = hh_qr_route(m, n, smem, batched=False)
    assert route == ("small" if m * n <= 4096 else "blocked")
    A = np.random.default_rng(m * 7919 + n).standard_normal((m, n))
    for label, Ai in edge_variants(A):
        (Q, R), nl = counted(ctx, lb.householder_qr, Ai, ctx=ctx)
        assert_route(route, nl, 1)
        check_householder(label, Ai, Q, R)


def test_max_cluster_is_measured_when_the_context_is_created(ctx):
    """A fresh context reports the panel kernel's largest cluster from the start, the same as one that has just run a
    blocked QR (1000 x 1000, beyond the one-CTA kernel), and a B200 holds clusters of at least 2 CTAs."""
    A = np.random.default_rng(1000).standard_normal((1000, 1000))
    lb.householder_qr(A, ctx=ctx)
    fresh = _native.Context(ctx.device)
    try:
        assert fresh.props()["max_cluster"] == ctx.props()["max_cluster"] >= 2
    finally:
        fresh.close()


def test_householder_qr_two_column_ranges_unpadded(ctx, smem):
    """2100 x 2017: 2048 padded columns, so Q is formed in two column ranges on two streams and then unpadded.  R against
    LAPACK (mode "r"; the reference's convention equals LAPACK's here because m > n, so no last row is negated), every
    diagonal sign, and the Q invariants."""
    m, n = 2100, 2017
    A = np.random.default_rng(2017).standard_normal((m, n))
    (Q, R), nl = counted(ctx, lb.householder_qr, A, ctx=ctx)
    assert_route(hh_qr_route(m, n, smem, batched=False), nl, 1)
    Rl = np.linalg.qr(A, mode="r")
    if m == n:
        Rl[-1] *= -1.0
    assert np.array_equal(np.sign(np.diag(R)), np.sign(np.diag(Rl)))
    assert orc.rel_max_err(R, Rl) <= REL
    assert np.all(np.tril(R, -1) == 0.0)
    assert orc.qr_residual(A, Q, R) <= RESID and orc.orth_error(Q) <= ORTH


@pytest.mark.parametrize("side", [0, 1], ids=["last_small", "first_blocked"])
@pytest.mark.parametrize("family", ["hh_square", "hh_tall2"])
def test_householder_qr_batched_smem_boundary(ctx, smem, family, side):
    """householder_qr_batched and its device-pointer form on both sides of the one-CTA shared-memory limit: beyond it each
    matrix runs through the blocked path (host entry: the one-matrix entry point; device entry: the blocked QR)."""
    m, n = boundary(family, smem)[side]
    route = hh_qr_route(m, n, smem, batched=True)
    assert route == ("small", "blocked")[side]
    rng = np.random.default_rng(m * 31 + n)
    cases = [("normal", rng.standard_normal((m, n))) for _ in range(3)] + edge_variants(rng.standard_normal((m, n)))[1:]
    A = np.stack([a for _, a in cases])
    nb = len(A)
    (Q, R), nl = counted(ctx, lb.householder_qr_batched, A, ctx=ctx)
    assert_route(route, nl, nb)
    dA, dQ, dR = ctx.upload(A), ctx.alloc(A.nbytes), ctx.alloc(8 * nb * n * n)
    _, nl = counted(ctx, ctx.call, "lq_householder_qr_batched_dev", dA.ptr, nb, m, n, dQ.ptr, dR.ptr, 0)
    assert_route(route, nl, nb)
    Qd, Rd = ctx.download(dQ, (nb, m, n)), ctx.download(dR, (nb, n, n))
    if route in ONE_KERNEL:
        assert np.array_equal(Q, Qd) and np.array_equal(R, Rd)
    for i, (label, Ai) in enumerate(cases):
        Qo, Ro = (None, None) if label == "dependent" else ref_householder_qr(Ai)
        check_householder(label, Ai, Q[i], R[i], Qo, Ro)
        check_householder(label, Ai, Qd[i], Rd[i], Qo, Ro)


# ----------------------------------------------------------------------------- MGS QR
@pytest.mark.parametrize("reorth", [False, True])
@pytest.mark.parametrize("side", [0, 1], ids=["last_small", "first_large"])
@pytest.mark.parametrize("family", ["mgs_square", "mgs_tall2"])
def test_mgs_qr_smem_boundary(ctx, smem, family, side, reorth):
    """qr / qr_batched / the device-pointer form on both sides of the one-CTA limit (beyond: one launch per column)."""
    m, n = boundary(family, smem)[side]
    route = mgs_qr_route(m, n, smem)
    assert route == ("small", "large")[side]
    rng = np.random.default_rng(m * 17 + n + reorth)
    A0 = rng.standard_normal((m, n))
    A = np.stack([A0, rng.standard_normal((m, n)), 1e-9 * A0, 1e7 * A0])
    nb = len(A)
    Qo, Ro = orc.mgs_qr_batched(A, reorth=reorth)

    def check(Q, R):
        assert orc.rel_max_err(Q, Qo) <= REL
        if reorth:  # the second sweep's R (close to I), compared absolutely as for the reference's own tests
            assert np.max(np.abs(R - Ro)) <= 1e-10
        else:
            for i in range(nb):
                assert orc.rel_max_err(R[i], Ro[i]) <= REL and orc.qr_residual(A[i], Q[i], R[i]) <= RESID, i
        assert np.all(np.tril(R, -1) == 0.0)

    (Q, R), nl = counted(ctx, lb.qr_batched, A, reorth=reorth, ctx=ctx)
    assert_route(route, nl, nb)
    check(Q, R)
    (Q1, R1), nl = counted(ctx, lb.qr, A[0], reorth=reorth, ctx=ctx)
    assert_route(route, nl, 1)
    assert np.array_equal(Q1, Q[0]) and np.array_equal(R1, R[0])
    dA, dQ, dR, dI = ctx.upload(A), ctx.alloc(A.nbytes), ctx.alloc(8 * nb * n * n), ctx.alloc(4 * nb)
    _, nl = counted(ctx, ctx.call, "lq_mgs_qr_batched_dev", dA.ptr, nb, m, n, int(reorth), dQ.ptr, dR.ptr, dI.ptr)
    assert_route(route, nl, nb)
    assert np.array_equal(ctx.download(dQ, (nb, m, n)), Q) and np.array_equal(ctx.download(dR, (nb, n, n)), R)
    assert not ctx.download(dI, (nb,), dtype=np.int32).any()


@pytest.mark.parametrize("side", [0, 1], ids=["last_small", "first_large"])
def test_mgs_qr_dependence_report_at_smem_boundary(ctx, smem, side):
    """Matrix 2 of a batch of 3 has column 9 = 2 x column 3 (or a zero column 9): qr_batched raises, the device entry
    reports info[2] == 10 (1-based) and nothing for the other two matrices."""
    m, n = boundary("mgs_square", smem)[side]
    rng = np.random.default_rng(500 + side)
    for how in ("dependent", "zero"):
        A = rng.standard_normal((3, m, n))
        A[2][:, 9] = 2.0 * A[2][:, 3] if how == "dependent" else 0.0
        with pytest.raises(ValueError, match="linearly dependent"):
            lb.qr_batched(A, ctx=ctx)
        with pytest.raises(ValueError, match="linearly dependent"):
            lb.qr(A[2], ctx=ctx)
        dA, dQ, dR, dI = ctx.upload(A), ctx.alloc(A.nbytes), ctx.alloc(8 * 3 * n * n), ctx.alloc(12)
        _, nl = counted(ctx, ctx.call, "lq_mgs_qr_batched_dev", dA.ptr, 3, m, n, 0, dQ.ptr, dR.ptr, dI.ptr)
        assert_route(mgs_qr_route(m, n, smem), nl, 3)
        assert ctx.download(dI, (3,), dtype=np.int32).tolist() == [0, 0, 10], how


# ----------------------------------------------------------------------------- least squares
TILE_SHAPES = [(m, n, k) for n in (1, 8, 9, 57, 63, 64) for k in (1, 8, 9, 15, 16) for m in sorted({n, n + 1, 4096})]
STREAM_SHAPES = [(65, 64, 17), (1000, 64, 32), (200, 1, 17), (4096, 40, 24)]
ONE_CTA_SHAPES = [(70, 65, 1), (120, 64, 33), "hh_ls:0", "hh_ls:1", "mgs_ls:0", "mgs_ls:1"]
LARGE_SHAPES = [(700, 300, 3), (600, 257, 1), (520, 512, 2), (400, 100, 300)]
LS_SHAPES = TILE_SHAPES + STREAM_SHAPES + ONE_CTA_SHAPES + LARGE_SHAPES


def _shape_id(s):
    return s.replace(":", "_") if isinstance(s, str) else "x".join(map(str, s))


def _resolve(shape, smem):
    if isinstance(shape, str):
        name, side = shape.split(":")
        return boundary(name, smem)[int(side)]
    return shape


LS_ENTRY = {
    "hh": ("lq_lstsq_householder_batched_info_dev", lb.least_squares_householder_qr_batched, lb.least_squares_householder_qr),
    "mgs": ("lq_lstsq_mgs_batched_dev", lb.least_squares_qr_batched, lb.least_squares_qr),
}


@pytest.mark.parametrize("shape", LS_SHAPES, ids=_shape_id)
@pytest.mark.parametrize("method", ["hh", "mgs"])
def test_least_squares_routes(ctx, smem, method, shape):
    """Tile (n <= 64, nrhs <= 16), stream (Householder, nrhs <= 32: several 64-row blocks, ragged last block), one-CTA
    and large routes, including the first / last shape that fits one CTA, against the extended-precision solution.  The
    device entry, the host pipeline and the one-matrix entry point give the same bits on the one-kernel routes."""
    m, n, k = _resolve(shape, smem)
    route = lstsq_route(method, m, n, k, smem)
    A, B, Xhp = ls_systems(m, n, k)
    nb = len(A)
    dev, batched, single = LS_ENTRY[method]
    dA, dB, dX, dI = ctx.upload(A), ctx.upload(B), ctx.alloc(8 * nb * n * k), ctx.upload(np.full(nb, -1, np.int32))
    _, nl = counted(ctx, ctx.call, dev, dA.ptr, dB.ptr, nb, m, n, k, dX.ptr, dI.ptr)
    assert_route(route, nl, nb)
    X = ctx.download(dX, (nb, n, k))
    assert not ctx.download(dI, (nb,), dtype=np.int32).any()
    for s in range(nb):
        check_x(X[s], A[s], B[s], Xhp[s], method)
    Xh, nl = counted(ctx, batched, A, B, ctx=ctx)
    assert_route(route, nl, nb)
    x0, nl = counted(ctx, single, A[0], B[0], ctx=ctx)
    assert_route(route, nl, 1)
    if route in ONE_KERNEL:
        assert np.array_equal(Xh.reshape(nb, n, k), X) and np.array_equal(x0.reshape(n, k), X[0])
    else:
        for s in range(nb):
            check_x(Xh.reshape(nb, n, k)[s], A[s], B[s], Xhp[s], method)
        check_x(x0.reshape(n, k), A[0], B[0], Xhp[0], method)


SINGULAR_SHAPES = [((100, 20, 4), "tile"), ((1000, 64, 32), "stream"), ((120, 64, 33), "small"),
                   ((400, 100, 300), "large"), ((700, 300, 3), "large")]


@pytest.mark.parametrize("shape,route", SINGULAR_SHAPES, ids=[f"{r}_{_shape_id(s)}" for s, r in SINGULAR_SHAPES])
def test_least_squares_householder_singular_R_every_route(ctx, smem, shape, route):
    """An exactly zero column leaves R[j, j] == 0 and np.linalg.solve (linalg/qr.py:134) raises LinAlgError: so does
    every Householder route, one-matrix and batched, and the device entry reports 1 + the first such column while the
    other systems of the batch are still solved."""
    m, n, k = shape
    assert lstsq_route("hh", m, n, k, smem) == route
    rng = np.random.default_rng(m + n + k)
    A, B = rng.standard_normal((4, m, n)), rng.standard_normal((4, m, k))
    A[1][:, n - 1] = 0.0
    A[3][:, 0] = 0.0
    if n > 2:
        A[3][:, n // 2] = 0.0
    dA, dB, dX, dI = ctx.upload(A), ctx.upload(B), ctx.alloc(8 * 4 * n * k), ctx.upload(np.full(4, -1, np.int32))
    ctx.call("lq_lstsq_householder_batched_info_dev", dA.ptr, dB.ptr, 4, m, n, k, dX.ptr, dI.ptr)
    assert ctx.download(dI, (4,), dtype=np.int32).tolist() == [0, n, 0, 1]
    X = ctx.download(dX, (4, n, k))
    for s in (0, 2):
        check_x(X[s], A[s], B[s], hp_householder(A[s], B[s])[2], "hh")
    Xo = np.full((4, n, k), np.nan)
    with pytest.raises(np.linalg.LinAlgError):
        lb.least_squares_householder_qr_batched(A, B, out=Xo, ctx=ctx)
    assert np.array_equal(Xo[[0, 2]], X[[0, 2]])
    for s in (1, 3):
        with pytest.raises(np.linalg.LinAlgError):
            lb.least_squares_householder_qr(A[s], B[s], ctx=ctx)
    lb.least_squares_householder_qr(A[0], B[0], ctx=ctx)


@pytest.mark.parametrize("shape,route", [((100, 20, 4), "tile"), ((120, 64, 33), "small"), ((700, 300, 3), "large")],
                         ids=["tile", "small", "large"])
def test_least_squares_mgs_dependence_every_route(ctx, smem, shape, route):
    """A zero or an exactly dependent column raises ValueError (linalg/qr.py:40-41) on every MGS route; the device entry
    reports 1 + that column."""
    m, n, k = shape
    assert lstsq_route("mgs", m, n, k, smem) == route
    rng = np.random.default_rng(m * n + k)
    A, B = rng.standard_normal((3, m, n)), rng.standard_normal((3, m, k))
    A[1][:, n - 1] = 0.0
    A[2][:, n // 2] = 2.0 * A[2][:, 1]
    dA, dB, dX, dI = ctx.upload(A), ctx.upload(B), ctx.alloc(8 * 3 * n * k), ctx.upload(np.full(3, -1, np.int32))
    ctx.call("lq_lstsq_mgs_batched_dev", dA.ptr, dB.ptr, 3, m, n, k, dX.ptr, dI.ptr)
    assert ctx.download(dI, (3,), dtype=np.int32).tolist() == [0, n, n // 2 + 1]
    with pytest.raises(ValueError, match="linearly dependent"):
        lb.least_squares_qr_batched(A, B, ctx=ctx)
    for s in (1, 2):
        with pytest.raises(ValueError, match="linearly dependent"):
            lb.least_squares_qr(A[s], B[s], ctx=ctx)


# ----------------------------------------------------------------------------- host pipelines with several chunks
def _chunk_samples(batch, chunk):
    idx = set()
    for lo in range(0, batch, chunk):
        hi = min(batch, lo + chunk)
        idx |= {lo, hi - 1}
    return sorted(idx)


def test_host_pipeline_qr32_several_chunks(ctx):
    """householder_qr_batched and qr_batched on 32 x 32 with 2 chunks + 5 matrices: both lanes, a ragged last chunk (MGS:
    24580 bytes per matrix, so its chunk is not a power of two).  Same bits as the device entry, the first and last matrix
    of every chunk against the oracle, and a dependent matrix in the last chunk only makes qr_batched raise."""
    per_hh = 3 * 32 * 32 * 8
    batch = 2 * chunk_of(per_hh) + 5
    A = np.random.default_rng(32).standard_normal((batch, 32, 32))
    dA, dQ, dR, dI = ctx.upload(A), ctx.alloc(A.nbytes), ctx.alloc(A.nbytes), ctx.alloc(4 * batch)
    for name, per, fn, ref in (("hh", per_hh, lb.householder_qr_batched, orc.householder_qr_batched),
                               ("mgs", per_hh + 4, lb.qr_batched, orc.mgs_qr_batched)):
        chunk = chunk_of(per)
        (Q, R), nl = counted(ctx, fn, A, ctx=ctx)
        assert nl == -(-batch // chunk) == 3, (name, nl, chunk)
        if name == "hh":
            ctx.call("lq_householder_qr_batched_dev", dA.ptr, batch, 32, 32, dQ.ptr, dR.ptr, 0)
        else:
            ctx.call("lq_mgs_qr_batched_dev", dA.ptr, batch, 32, 32, 0, dQ.ptr, dR.ptr, dI.ptr)
        assert np.array_equal(Q, ctx.download(dQ, A.shape)) and np.array_equal(R, ctx.download(dR, A.shape)), name
        idx = _chunk_samples(batch, chunk)
        Qo, Ro = ref(A[idx])
        assert orc.rel_max_err(Q[idx], Qo) <= REL and orc.rel_max_err(R[idx], Ro) <= REL, name
    Ad = A.copy()
    Ad[batch - 2][:, 9] = 2.0 * Ad[batch - 2][:, 3]
    with pytest.raises(ValueError, match="linearly dependent"):
        lb.qr_batched(Ad, ctx=ctx)


@pytest.mark.parametrize("pinned", [False, True], ids=["pageable", "pinned"])
def test_host_pipeline_cfg3_several_chunks(ctx, pinned):
    """Both batched least-squares entry points on 256 x 64 with 16 right-hand sides and 2 chunks + 7 systems, from pageable
    and from page-locked buffers: same bits as the device entry, samples of every chunk against the extended-precision
    solution, and a zero column in the last chunk only raises (info offsets of the last chunk)."""
    m, n, k = 256, 64, 16
    per = 8 * (m * n + m * k + n * k) + 4
    chunk = chunk_of(per)
    batch = 2 * chunk + 7
    rng = np.random.default_rng(3)
    A, B = rng.standard_normal((batch, m, n)), rng.standard_normal((batch, m, k))
    if pinned:
        Ap, Bp = _native.pinned_empty(A.shape), _native.pinned_empty(B.shape)
        Ap[...], Bp[...] = A, B
        A, B = Ap, Bp
    dA, dB, dX, dI = ctx.upload(A), ctx.upload(B), ctx.alloc(8 * batch * n * k), ctx.alloc(4 * batch)
    idx = _chunk_samples(batch, chunk)
    for method in ("hh", "mgs"):
        dev, fn, _ = LS_ENTRY[method]
        out = _native.pinned_empty((batch, n, k)) if pinned else None
        X, nl = counted(ctx, fn, A, B, out=out, ctx=ctx)
        assert nl == -(-batch // chunk) == 3, (method, nl, chunk)
        ctx.call(dev, dA.ptr, dB.ptr, batch, m, n, k, dX.ptr, dI.ptr)
        assert np.array_equal(X.reshape(batch, n, k), ctx.download(dX, (batch, n, k))), method
        assert not ctx.download(dI, (batch,), dtype=np.int32).any()
        for s in idx:
            check_x(X.reshape(batch, n, k)[s], A[s], B[s], hp_householder(A[s], B[s])[2], method)
    As = np.array(A)
    As[batch - 3][:, 17] = 0.0
    with pytest.raises(np.linalg.LinAlgError):
        lb.least_squares_householder_qr_batched(As, B, ctx=ctx)
    with pytest.raises(ValueError, match="linearly dependent"):
        lb.least_squares_qr_batched(As, B, ctx=ctx)

"""Every entry point under power-of-two scaling of its input, across the exponent range.

Scaling by s = 4^j is exact in floating point.  As long as no intermediate leaves the normal range and no absolute
threshold is crossed, the same sums are formed in the same order, FMA and DMMA round the same way, and the MUFU seeds and
their Newton steps scale exactly (the rsqrt seed depends on the parity of the exponent, hence even powers of two).  So
every output must scale by its known power of two BIT FOR BIT: this compares each kernel with itself over about 2000
binades, and together with the unit-scale accuracy the route suites prove (``test_gpu_routes.py``,
``test_gpu_tallskinny_routes.py``) gives accuracy at every scale.  An absolute constant hidden in a kernel fails it.

- QR and MGS: (Q, R)(sA) = (Q, sR); least squares: X(sA, tB) = (t / s) X(A, B); tsqr: (Q, sR); Gram: G(sA) = s^2 G(A);
  eigen-solver: eigh(sG) = (s lambda, V); svd(sA) = (U, s sigma, Vt); GEMM: C(sA, tB, beta, st C0) = st C(A, B, beta, C0);
  pca: pcs and ratios unchanged, scores x s, variances x s^2; projection: P(sA, tb) = t P(A, b); det(sA) = s^n det(A).
- Sweep: QR, MGS, least squares, tsqr and det keep every R[j, j] >= 2^-20 (well above the reference's absolute 1e-12) and
  every column norm <= 2^480 (NumPy's norm overflows from 2^512).  The Gram, eigen-solver, SVD and pca families take max
  diag(A^T A) from 2^-900 to 2^960 (below about 2^-1000 single products a_ik a_jk are subnormal).
- At the smallest and largest scale of each family the result is also held to the plain reference at the bars the route
  suites use.  Where the reference's absolute thresholds act, the result must follow the reference's decision instead
  (a column norm of 1e-12 (1 +- 2^-20) on every Householder and MGS route; an all-zero matrix through svd and eigh).
"""
import math

import numpy as np
import pytest

import linalg_b200 as lb
from oracle import linalg_oracle as orc
from test_gpu_routes import (U64, _hp, _hp_sqrt, assert_route, check_x, conditioned, counted, hh_qr_route, hp_householder,
                             lstsq_route, mgs_qr_route, ref_householder_qr)
from test_gpu_tallskinny_routes import (C_TSQR, REL, eig_errors, eigh_route, gram_route, replay_vt, svd_errors, svd_route,
                                        tsqr_route, with_option)

pytestmark = pytest.mark.gpu

R_MIN_LOG2 = -20     # smallest |R[j, j]| of the QR-type sweeps
NORM_MAX_LOG2 = 480  # largest column norm of the QR-type sweeps
GRAM_LOG2 = (-900, 960)  # range of max diag(A^T A) of the Gram-type sweeps


def sc(x, j):
    """x * 4^j, exactly."""
    return np.ldexp(x, 2 * j)


def log2(x):
    return math.log2(float(x))


def qr_bounds(A):
    """Range of j (s = 4^j) that keeps every |R[j, j]| of every matrix of A >= 2^-20 and every column norm <= 2^480."""
    A = A.reshape((-1,) + A.shape[-2:])
    dmin = min(np.min(np.abs(np.diag(np.linalg.qr(a, mode="r")))) for a in A)
    cmax = np.max(np.linalg.norm(A, axis=-2))
    return math.ceil((R_MIN_LOG2 - log2(dmin)) / 2), math.floor((NORM_MAX_LOG2 - log2(cmax)) / 2)


def qr_js(A):
    return spread(*qr_bounds(A))


def gram_js(dmax, per_j=4):
    """Exponents j that put max diag (scaled by 2^(per_j j)) in the Gram-type range."""
    lo = math.ceil((GRAM_LOG2[0] - log2(dmax)) / per_j)
    hi = math.floor((GRAM_LOG2[1] - log2(dmax)) / per_j)
    return spread(lo, hi)


def spread(lo, hi):
    assert lo < -1 and hi > 1, (lo, hi)
    return sorted({lo, lo // 2, -1, 1, hi // 2, hi})


def same(label, got, want):
    assert got.shape == want.shape and np.array_equal(got, want), (label, np.max(np.abs(got - want)))


# ----------------------------------------------------------------------------- Householder QR
# (label, shape of the batch, batched): one representative shape per route; the mirrors of test_gpu_routes name the route
HH_CASES = [("small", (3, 40, 24), True), ("qr32", (3, 32, 32), True), ("blocked_batched", (2, 169, 169), True),
            ("one_cta", (1, 64, 64), False), ("blocked", (1, 255, 200), False)]


@pytest.mark.parametrize("label,shape,batched", HH_CASES, ids=[c[0] for c in HH_CASES])
def test_householder_qr_scaling(ctx, label, shape, batched):
    nb, m, n = shape
    smem = ctx.props()["max_smem"]
    route = hh_qr_route(m, n, smem, batched)
    A = np.random.default_rng(m * n + nb).standard_normal(shape)

    def run(X):
        if batched:
            (Q, R), nl = counted(ctx, lb.householder_qr_batched, X, ctx=ctx)
        else:
            (Q, R), nl = counted(ctx, lb.householder_qr, X[0], ctx=ctx)
            Q, R = Q[None], R[None]
        assert_route(route, nl, nb)
        return Q, R

    Q0, R0 = run(A)
    js = qr_js(A)
    for j in js:
        Q, R = run(sc(A, j))
        same(f"{label} Q j={j}", Q, Q0)
        same(f"{label} R j={j}", R, sc(R0, j))
        if j in (js[0], js[-1]):
            for i in range(nb):
                Qo, Ro = ref_householder_qr(sc(A[i], j))
                assert orc.rel_max_err(Q[i], Qo) <= REL and orc.rel_max_err(R[i], Ro) <= REL, (label, j, i)


# ----------------------------------------------------------------------------- MGS QR
MGS_CASES = [("small", (3, 40, 24)), ("qr32", (3, 32, 32)), ("large", (2, 121, 121))]


@pytest.mark.parametrize("label,shape", MGS_CASES, ids=[c[0] for c in MGS_CASES])
def test_mgs_qr_scaling(ctx, label, shape):
    nb, m, n = shape
    route = mgs_qr_route(m, n, ctx.props()["max_smem"])
    A = np.random.default_rng(7 * m + n).standard_normal(shape)

    def run(X):
        (Q, R), nl = counted(ctx, lb.qr_batched, X, ctx=ctx)
        assert_route(route, nl, nb)
        (Q1, R1), nl = counted(ctx, lb.qr, X[0], ctx=ctx)
        assert_route(route, nl, 1)
        same("qr vs qr_batched", Q1, Q[0])
        same("qr vs qr_batched", R1, R[0])
        return Q, R

    Q0, R0 = run(A)
    js = qr_js(A)
    for j in js:
        Q, R = run(sc(A, j))
        same(f"{label} Q j={j}", Q, Q0)
        same(f"{label} R j={j}", R, sc(R0, j))
        if j in (js[0], js[-1]):
            Qo, Ro = orc.mgs_qr_batched(sc(A, j))
            assert orc.rel_max_err(Q, Qo) <= REL and orc.rel_max_err(R, Ro) <= REL, (label, j)


# ----------------------------------------------------------------------------- least squares
LS_CASES = [("hh", "tile", (100, 20, 4)), ("hh", "stream", (1000, 64, 32)), ("hh", "small", (120, 64, 33)),
            ("hh", "large", (600, 257, 1)), ("mgs", "tile", (100, 20, 4)), ("mgs", "small", (120, 64, 33)),
            ("mgs", "large", (600, 257, 1))]
LS_ENTRY = {"hh": ("lq_lstsq_householder_batched_info_dev", lb.least_squares_householder_qr_batched),
            "mgs": ("lq_lstsq_mgs_batched_dev", lb.least_squares_qr_batched)}


@pytest.mark.parametrize("method,route,shape", LS_CASES, ids=[f"{m}_{r}" for m, r, _ in LS_CASES])
def test_least_squares_scaling(ctx, method, route, shape):
    m, n, k = shape
    assert lstsq_route(method, m, n, k, ctx.props()["max_smem"]) == route
    rng = np.random.default_rng(m + 3 * n + k)
    A = np.stack([rng.standard_normal((m, n)), conditioned(rng, m, n, 1e3)])
    B = rng.standard_normal((2, m, k))
    nb = len(A)
    dev, host = LS_ENTRY[method]

    def run(As, Bs):
        dA, dB, dX, dI = ctx.upload(As), ctx.upload(Bs), ctx.alloc(8 * nb * n * k), ctx.upload(np.full(nb, -1, np.int32))
        _, nl = counted(ctx, ctx.call, dev, dA.ptr, dB.ptr, nb, m, n, k, dX.ptr, dI.ptr)
        assert_route(route, nl, nb)
        assert not ctx.download(dI, (nb,), dtype=np.int32).any()
        X = ctx.download(dX, (nb, n, k))
        if route in ("tile", "stream", "small"):
            same("host pipeline", np.asarray(host(As, Bs, ctx=ctx)).reshape(nb, n, k), X)
        return X

    X0 = run(A, B)
    js = qr_js(A)
    bmax = log2(np.max(np.linalg.norm(B, axis=-2)))
    for j in js:
        for jt in sorted({j, -j, 0}):
            if 2 * jt + bmax > NORM_MAX_LOG2:
                continue
            X = run(sc(A, j), sc(B, jt))
            same(f"{method} {route} j={j} jt={jt}", X, sc(X0, jt - j))
            if jt == j and j in (js[0], js[-1]):
                As, Bs = sc(A, j), sc(B, j)
                for s in range(nb):
                    check_x(X[s], As[s], Bs[s], hp_householder(As[s], Bs[s])[2], method)


# ----------------------------------------------------------------------------- tsqr
TSQR_CASES = [("cholqr2", (4000, 40)), ("bcgs2", (1000, 130)), ("householder", (100, 40))]


@pytest.mark.parametrize("route,shape", TSQR_CASES, ids=[c[0] for c in TSQR_CASES])
def test_tsqr_scaling(ctx, route, shape):
    m, n = shape
    assert tsqr_route(m, n) == route
    A = np.random.default_rng(m + n).standard_normal((m, n))
    Q0, R0 = lb.tsqr(A, ctx=ctx)
    Qh, Rh = with_option(ctx, "TSQR_HOUSEHOLDER", lb.tsqr, A)
    assert (np.array_equal(Q0, Qh) and np.array_equal(R0, Rh)) == (route == "householder"), route
    js = qr_js(A)
    kappa = np.linalg.cond(A)
    for j in js:
        Q, R = lb.tsqr(sc(A, j), ctx=ctx)
        same(f"tsqr {route} Q j={j}", Q, Q0)
        same(f"tsqr {route} R j={j}", R, sc(R0, j))
        if j in (js[0], js[-1]):
            _, Ro = orc.tsqr_reference(sc(A, j))
            err = orc.rel_max_err(R, Ro)
            assert err <= C_TSQR * max(m, n) * U64 * kappa and err <= REL, (route, j, err)


# ----------------------------------------------------------------------------- Gram matrix
GRAM_CASES = [("syrk", (2048, 64)), ("gemm", (1023, 128))]


@pytest.mark.parametrize("route,shape", GRAM_CASES, ids=[c[0] for c in GRAM_CASES])
def test_gram_scaling(ctx, route, shape):
    m, n = shape
    assert gram_route(m, n) == route
    Ai = np.random.default_rng(m + n).integers(-1024, 1025, size=(m, n)).astype(np.float64)
    exact = (Ai.astype(np.int64).T @ Ai.astype(np.int64)).astype(np.float64)

    def run(A):
        dA, dG, dH = ctx.upload(A), ctx.alloc(8 * n * n), ctx.alloc(8 * n * n)
        _, nl = counted(ctx, ctx.call, "lq_gram_dev", dA.ptr, m, n, dG.ptr)
        ctx.call("lq_gemm_dev", 1, 0, n, n, m, 1.0, dA.ptr, n, dA.ptr, n, 0.0, dH.ptr, n)
        G, H = ctx.download(dG, (n, n)), ctx.download(dH, (n, n))
        assert (nl == 2 and not np.array_equal(G, H)) if route == "syrk" else np.array_equal(G, H), (route, nl)
        return G

    A = np.random.default_rng(m * n).standard_normal((m, n))
    G0 = run(A)
    js = gram_js(np.max(np.diag(G0)))
    for j in js:
        same(f"gram {route} j={j}", run(sc(A, j)), sc(G0, 2 * j))
        if j in (js[0], js[-1]):   # integer input: every partial sum is exact, at every scale
            dA, dG = ctx.upload(sc(Ai, j)), ctx.alloc(8 * n * n)
            ctx.call("lq_gram_dev", dA.ptr, m, n, dG.ptr)
            same(f"gram {route} integer j={j}", ctx.download(dG, (n, n)), sc(exact, 2 * j))


# ----------------------------------------------------------------------------- eigen-solver
EIG_CASES = [("one_sided_0", 64), ("one_sided_8", 128), ("two_sided_smem", 150), ("two_sided_global", 200)]


def eigh(ctx, G):
    n = G.shape[0]
    dG, dl, dV = ctx.upload(G), ctx.alloc(8 * n), ctx.alloc(8 * n * n)
    _, nl = counted(ctx, ctx.call, "lq_eigh_dev", dG.ptr, n, dl.ptr, dV.ptr)
    return ctx.download(dl, (n,)), ctx.download(dV, (n, n)), nl


@pytest.mark.parametrize("route,n", EIG_CASES, ids=[c[0] for c in EIG_CASES])
def test_eigh_scaling(ctx, route, n):
    """The one-sided solver used to stop rotating once max diag(G) left 2^-256 .. 2^256 (its rotation test multiplies four
    entries), the two-sided one above 2^512: both now work on G scaled to a unit diagonal."""
    assert eigh_route(n, ctx.props()["max_smem"]) == route
    M = np.random.default_rng(n).standard_normal((n + 7, n))
    G = M.T @ M
    lam0, V0, nl = eigh(ctx, G)
    assert nl == (4 if route.startswith("one_sided") else 3), (route, nl)
    js = gram_js(np.max(np.diag(G)), per_j=2)
    for j in js:
        lam, V, _ = eigh(ctx, sc(G, j))
        same(f"eigh {route} lambda j={j}", lam, sc(lam0, j))
        same(f"eigh {route} V j={j}", V, V0)
        if j in (js[0], js[-1]):   # LAPACK on the scaled matrix; the checks are homogeneous, so compare at unit scale
            lr, Vr = np.linalg.eigh(sc(G, j))
            assert_ok(f"eigh {route} j={j}", eig_errors(G, sc(lam, -j), V, sc(lr, -j), Vr))


def assert_ok(label, checks):
    ratios = {k: float(e / b) if b > 0 else (0.0 if e == 0 else np.inf) for k, (e, b) in checks.items()}
    assert all(r <= 1.0 for r in ratios.values()), (label, ratios)


def test_eigh_zero_matrix(ctx):
    """max diag = 0: no scaling, lambda = 0 and V = I on both kernels."""
    for n in (64, 128, 150, 200):
        lam, V, _ = eigh(ctx, np.zeros((n, n)))
        assert np.all(lam == 0.0) and np.isfinite(V).all() and np.max(np.abs(V.T @ V - np.eye(n))) <= 1e-12, n


# ----------------------------------------------------------------------------- SVD
SVD_CASES = [("direct", (3000, 64), "gaussian"), ("replay", (3000, 64), "kappa1e4"), ("two_sided", (1500, 200), "gaussian")]


@pytest.mark.parametrize("route,shape,spectrum", SVD_CASES, ids=[c[0] for c in SVD_CASES])
def test_svd_scaling(ctx, route, shape, spectrum):
    """tol = 0 keeps U = A V / s at every scale, so all three factors are compared bitwise.  At the small end the default
    tol = 1e-12 exceeds every sigma: s and Vt stay the same, U is the seeded completion (orthonormal, rank 0)."""
    m, n = shape
    rng = np.random.default_rng(m + n)
    A = rng.standard_normal((m, n)) if spectrum == "gaussian" else conditioned(rng, m, n, float(spectrum[5:]))
    sigma = np.linalg.svd(A, compute_uv=False)
    assert (svd_route(n, sigma) if n <= 128 else "two_sided") == route
    U0, s0, Vt0 = lb.svd(A, 0.0, ctx=ctx)
    if n <= 128:
        assert np.array_equal(Vt0, replay_vt(ctx, A)[0]) == (route == "replay"), route
    js = gram_js(sigma[0] ** 2)
    for j in js:
        U, s, Vt = lb.svd(sc(A, j), 0.0, ctx=ctx)
        same(f"svd {route} U j={j}", U, U0)
        same(f"svd {route} s j={j}", s, sc(s0, j))
        same(f"svd {route} Vt j={j}", Vt, Vt0)
        if j in (js[0], js[-1]):
            _, sr, Vtr = np.linalg.svd(sc(A, j), full_matrices=False)
            assert_ok(f"svd {route} j={j}", svd_errors(A, U, sc(s, -j), Vt, sc(sr, -j), Vtr.T))
    j = js[0]
    U, s, Vt = lb.svd(sc(A, j), ctx=ctx, seed=5)
    assert np.max(s) <= 1e-12
    same("svd default tol s", s, sc(s0, j))
    same("svd default tol Vt", Vt, Vt0)
    assert np.max(np.abs(U.T @ U - np.eye(n))) <= 1e-12


@pytest.mark.parametrize("shape", [(300, 64), (300, 128), (400, 150), (400, 200)], ids=lambda s: f"{s[0]}x{s[1]}")
def test_svd_zero_matrix(ctx, shape):
    """An all-zero matrix: the eigen-solver sees max diag = 0 and must not scale; s = 0, rank 0, finite orthonormal U."""
    m, n = shape
    U, s, Vt = lb.svd(np.zeros((m, n)), ctx=ctx, seed=3)
    assert np.all(s == 0.0) and np.isfinite(U).all() and np.isfinite(Vt).all()
    assert np.max(np.abs(U.T @ U - np.eye(n))) <= 1e-12 and np.max(np.abs(Vt @ Vt.T - np.eye(n))) <= 1e-12


# ----------------------------------------------------------------------------- GEMM
def gemm_route(ta, tb, M, N, K, beta, sms):
    """Mirror of gemm() (gemm.cu): generic, update (NN, K % 16 == 0, beta in {0, 1}, >= 2 sm_count 128 x 64 tiles),
    rank (NN, 16 <= K <= 128, M >= 256, < 4 column tiles, >= 4 row tiles), split-K (< 2 sm_count tiles, >= 16 k-tiles),
    fast, and fast + generic for a K remainder."""
    Km = K - K % 16
    fast = Km >= 16 and M * N >= 1024 and (M % 2 == 0 or not ta) and (N % 2 == 0 or tb)
    if not fast:
        return "generic"
    tm, tn = -(-M // 128), -(-N // 128)
    if not ta and not tb and Km == K:
        if beta in (0.0, 1.0) and N % 2 == 0 and M >= 128 and N >= 64 and K <= 512 and tm * (-(-N // 64)) >= 2 * sms:
            return "update"
        if K <= 128 and N % 2 == 0 and M >= 256 and tn < 4 and tm >= 4:
            return "rank"
    if Km < K:
        return "remainder"
    return "split" if tm * tn < 2 * sms and Km // 16 >= 16 else "fast"


GEMM_CASES = [("generic", 0, 0, (20, 30, 40)), ("fast_nn", 0, 0, (256, 192, 64)), ("fast_tn", 1, 0, (256, 192, 64)),
              ("fast_nt", 0, 1, (256, 192, 64)), ("fast_tt", 1, 1, (256, 192, 64)), ("update", 0, 0, (2560, 1024, 64)),
              ("rank", 0, 0, (4096, 128, 128)), ("split", 1, 0, (64, 64, 4096)), ("remainder", 0, 1, (300, 200, 100))]
GEMM_SCALES = [(-220, -220), (-240, 240), (240, -240), (230, 230), (7, -3)]


@pytest.mark.parametrize("label,ta,tb,shape", GEMM_CASES, ids=[c[0] for c in GEMM_CASES])
def test_gemm_scaling(ctx, label, ta, tb, shape):
    M, N, K = shape
    sms = ctx.props()["sm_count"]
    rng = np.random.default_rng(M + N + K)
    A = rng.standard_normal((K, M) if ta else (M, K))
    B = rng.standard_normal((N, K) if tb else (K, N))
    C0 = rng.standard_normal((M, N))
    opA, opB = (A.T if ta else A), (B.T if tb else B)

    def run(As, Bs, Cs, alpha, beta):
        dA, dB, dC = ctx.upload(As), ctx.upload(Bs), ctx.upload(Cs)
        _, nl = counted(ctx, ctx.call, "lq_gemm_dev", ta, tb, M, N, K, alpha, dA.ptr, As.shape[1], dB.ptr, Bs.shape[1], beta,
                        dC.ptr, N)
        route = gemm_route(ta, tb, M, N, K, beta, sms)
        assert nl == (2 if route in ("split", "remainder") else 1), (route, nl)
        return ctx.download(dC, (M, N)), route

    P = opA @ opB
    absP = np.abs(opA) @ np.abs(opB)
    routes = set()
    for alpha in (0.0, 1.0, -0.75):
        for beta in (0.0, 1.0, 0.375):
            Cu, route = run(A, B, C0, alpha, beta)
            routes.add(route)
            for j, k in GEMM_SCALES:
                C, _ = run(sc(A, j), sc(B, k), sc(C0, j + k), alpha, beta)
                same(f"gemm {label} alpha={alpha} beta={beta} j={j} k={k}", C, sc(Cu, j + k))
                if (j, k) == GEMM_SCALES[0]:   # against the float64 product: twice the bound, for the reference's rounding
                    err = np.abs(sc(C, -j - k) - (alpha * P + beta * C0))
                    assert np.all(err <= 4 * K * U64 * (abs(alpha) * absP + abs(beta) * np.abs(C0))), (label, alpha, beta)
    # the update kernel takes beta in {0, 1} only; the other beta runs on the generic tensor-core kernel
    assert routes == ({"update", "fast"} if label == "update" else {label.split("_")[0]}), (label, routes)


# ----------------------------------------------------------------------------- pca, projection, det / adj
@pytest.mark.parametrize("shape", [(2000, 48), (600, 150)], ids=["one_sided", "two_sided"])
def test_pca_scaling(ctx, shape):
    m, n = shape
    A = np.random.default_rng(n).standard_normal((m, n)) + 3.0
    k = 5
    pcs0, sc0, ev0, r0, tv0, mu0 = lb.pca(A, k, ctx=ctx)
    X = A - A.mean(axis=0)
    js = gram_js(np.max(np.sum(X * X, axis=0)))
    for j in js:
        pcs, scr, ev, r, tv, mu = lb.pca(sc(A, j), k, ctx=ctx)
        same(f"pca pcs j={j}", pcs, pcs0)
        same(f"pca ratio j={j}", r, r0)
        same(f"pca scores j={j}", scr, sc(sc0, j))
        same(f"pca variance j={j}", ev, sc(ev0, 2 * j))
        assert tv == math.ldexp(tv0, 4 * j) and np.array_equal(mu, sc(mu0, j)), j
        if j in (js[0], js[-1]):
            sv = np.linalg.svd(sc(X, j), compute_uv=False)
            ev_ref = sc(sv[:k], -j) ** 2 / (m - 1)
            assert np.max(np.abs(sc(ev, -2 * j) - ev_ref) / ev_ref) <= 1e-10, j


def hp_projection(A, b):
    """A (A^T A)^-1 A^T b in extended precision (full column rank)."""
    Ah, bh = _hp(A), _hp(b)
    G, y = Ah.T @ Ah, Ah.T @ bh
    n = G.shape[0]
    L = np.zeros_like(G)
    for i in range(n):   # Cholesky G = L L^T
        for k in range(i + 1):
            v = G[i, k] - L[i, :k] @ L[k, :k]
            L[i, k] = _hp_sqrt(v) if i == k else v / L[k, k]
    z = y.copy()
    for i in range(n):
        z[i] = (z[i] - L[i, :i] @ z[:i]) / L[i, i]
    for i in range(n - 1, -1, -1):
        z[i] = (z[i] - L[i + 1:, i] @ z[i + 1:]) / L[i, i]
    return (Ah @ z).astype(np.float64)


PROJ_CASES = [("qr", (50, 3)), ("qr", (200, 20)), ("svd", (60, 5))]


@pytest.mark.parametrize("branch,shape", PROJ_CASES, ids=[f"{b}_{m}x{n}" for b, (m, n) in PROJ_CASES])
def test_project_onto_colspace_scaling(ctx, branch, shape):
    """Scale-invariant like the reference's normal equations: down to 4^-200 (column norms far below the QR's absolute
    1e-12 skip, which used to send the Q branch to columns of the identity) and up to 4^200."""
    m, n = shape
    rng = np.random.default_rng(m * n)
    A = rng.standard_normal((m, n))
    if branch == "svd":
        A[:, n - 1] = A[:, 0] - 0.5 * A[:, 1]
    b = rng.standard_normal((m, 2))
    P0 = lb.project_onto_colspace(A, b, ctx=ctx)
    Aind = A[:, :n - 1] if branch == "svd" else A
    js = [-200, -22, -7, -1, 1, 7, 200]
    for j in js:
        for jt in sorted({j, -j, 0}):
            same(f"projection {branch} j={j} jt={jt}", lb.project_onto_colspace(sc(A, j), sc(b, jt), ctx=ctx), sc(P0, jt))
        if j in (js[0], js[-1]):
            P = lb.project_onto_colspace(sc(A, j), sc(b, j), ctx=ctx)
            ref = hp_projection(sc(Aind, j), sc(b, j))
            err = np.linalg.norm(P - ref, axis=0) / np.linalg.norm(ref, axis=0)
            assert np.max(err) <= 64 * m * U64, (branch, j, err)


@pytest.mark.parametrize("n", [6, 32])
def test_det_adj_scaling(ctx, n):
    """det(sA) = s^n det(A) and adj(sA) = s^(n - 1) adj(A) through the batched Householder QR (small and 32 x 32 routes)."""
    A = np.random.default_rng(n).standard_normal((4, n, n))
    d0 = lb.det_batched(A, ctx=ctx)
    a0 = lb.adj_batched(A, ctx=ctx)
    lo, hi = qr_bounds(A)
    ld, la = np.log2(np.abs(d0)), np.log2(np.abs(a0[a0 != 0]))
    lo = max(lo, math.ceil((-1000 - ld.min()) / (2 * n)), math.ceil((-1000 - la.min()) / (2 * (n - 1))))
    hi = min(hi, math.floor((1000 - ld.max()) / (2 * n)), math.floor((1000 - la.max()) / (2 * (n - 1))))
    js = spread(lo, hi)
    for j in js:
        d = lb.det_batched(sc(A, j), ctx=ctx)
        same(f"det n={n} j={j}", d, np.ldexp(d0, 2 * j * n))
        same(f"adj n={n} j={j}", lb.adj_batched(sc(A, j), ctx=ctx), sc(a0, j * (n - 1)))
    for j in (js[0], js[-1]):
        d = lb.det_batched(sc(A, j), ctx=ctx)
        ref = np.linalg.det(sc(A, j))
        assert np.max(np.abs(d - ref) / np.abs(ref)) <= 1e-10, (n, j)


# ----------------------------------------------------------------------------- the absolute threshold, 1e-12
def threshold_matrix(rng, m, n, col, factor):
    """Gaussian columns, and column `col` exactly orthogonal to the others with norm 1e-12 * factor: its remaining norm
    when the factorisation reaches it is that norm (to rounding, far inside 2^-20)."""
    W = rng.standard_normal((m, n))
    others = np.delete(W, col, axis=1)
    Qo, _ = np.linalg.qr(others, mode="complete")
    c = Qo[:, n - 1:] @ rng.standard_normal(m - n + 1)
    W[:, col] = c / np.linalg.norm(c) * (orc.EPS * factor)
    return W


FACTORS = {"above": 1 + 2.0 ** -20, "below": 1 - 2.0 ** -20}
THRESH_QR = [("hh", "small", (40, 24), True), ("hh", "qr32", (32, 32), True), ("hh", "blocked", (169, 169), True),
             ("hh", "small", (64, 64), False), ("hh", "blocked", (255, 200), False),
             ("mgs", "small", (40, 24), True), ("mgs", "qr32", (32, 32), True), ("mgs", "large", (121, 121), True)]


@pytest.mark.parametrize("side", list(FACTORS))
@pytest.mark.parametrize("method,route,shape,batched", THRESH_QR, ids=[f"{m}_{r}_{'batched' if b else 'single'}" for m, r, _, b in THRESH_QR])
def test_qr_threshold_decision(ctx, method, route, shape, batched, side):
    """A column of norm 1e-12 (1 +- 2^-20), first and last: Householder applies / skips its reflector exactly when the
    oracle does (Q against the oracle at 1e-10), MGS raises exactly when the oracle does."""
    m, n = shape
    smem = ctx.props()["max_smem"]
    assert (hh_qr_route(m, n, smem, batched) if method == "hh" else mgs_qr_route(m, n, smem)) == route
    rng = np.random.default_rng(m + n)
    A = np.stack([threshold_matrix(rng, m, n, col, FACTORS[side]) for col in (0, n - 1)])
    if method == "hh":
        if batched:
            (Q, R), nl = counted(ctx, lb.householder_qr_batched, A, ctx=ctx)
            assert_route(route, nl, len(A))
        else:
            outs = [counted(ctx, lb.householder_qr, a, ctx=ctx) for a in A]
            for _, nl in outs:
                assert_route(route, nl, 1)
            Q, R = np.stack([q for (q, _), _ in outs]), np.stack([r for (_, r), _ in outs])
        for i in range(len(A)):
            Qo, Ro = ref_householder_qr(A[i])
            assert orc.rel_max_err(Q[i], Qo) <= REL and orc.rel_max_err(R[i], Ro) <= REL, (route, side, i)
        return
    for i in range(len(A)):
        try:
            orc.mgs_qr(A[i])
            raised = False
        except ValueError:
            raised = True
        assert raised == (side == "below")
        if raised:
            with pytest.raises(ValueError, match="linearly dependent"):
                lb.qr_batched(A[i:i + 1], ctx=ctx)
        else:
            (Q, R), nl = counted(ctx, lb.qr_batched, A[i:i + 1], ctx=ctx)
            assert_route(route, nl, 1)
            Qo, Ro = orc.mgs_qr(A[i])
            assert orc.rel_max_err(Q[0], Qo) <= REL, (route, side, i)


THRESH_LS = [("hh", "tile", (100, 20, 4)), ("hh", "stream", (1000, 64, 32)), ("hh", "small", (120, 64, 33)),
             ("hh", "large", (600, 257, 1)), ("mgs", "tile", (100, 20, 4)), ("mgs", "small", (120, 64, 33)),
             ("mgs", "large", (600, 257, 1))]


@pytest.mark.parametrize("side", list(FACTORS))
@pytest.mark.parametrize("method,route,shape", THRESH_LS, ids=[f"{m}_{r}" for m, r, _ in THRESH_LS])
def test_least_squares_threshold_decision(ctx, method, route, shape, side):
    """The same columns through least squares.  MGS: info exactly when the oracle raises (every route).  Householder:
    nothing is raised on either side (the reference's skip leaves R[j, j] = x[0] != 0), and X follows the extended-precision
    factorisation row by row to 1e-6 of that row's size (applying or skipping gives O(1) different solutions).  Above the
    threshold every route applies the reflector, as the reference does.  Below it the one-CTA routes skip it like the
    reference; the tile and stream routes factor row blocks and carry only R, so no block sees the whole column: they skip
    exactly zero columns only (skipping a block's part would drop its rows, and a column of norm 1.5e-12 spread over the
    blocks ended with R[j, j] = 0, a LinAlgError the reference does not raise), and match the applied factorisation."""
    m, n, k = shape
    assert lstsq_route(method, m, n, k, ctx.props()["max_smem"]) == route
    rng = np.random.default_rng(m * k + n)
    A = np.stack([threshold_matrix(rng, m, n, col, FACTORS[side]) for col in (0, n - 1)])
    B = rng.standard_normal((2, m, k))
    dev, _ = LS_ENTRY[method]
    dA, dB, dX, dI = ctx.upload(A), ctx.upload(B), ctx.alloc(8 * 2 * n * k), ctx.upload(np.full(2, -1, np.int32))
    _, nl = counted(ctx, ctx.call, dev, dA.ptr, dB.ptr, 2, m, n, k, dX.ptr, dI.ptr)
    assert_route(route, nl, 2)
    info = ctx.download(dI, (2,), dtype=np.int32)
    X = ctx.download(dX, (2, n, k))
    if method == "mgs":
        assert info.tolist() == ([1, n] if side == "below" else [0, 0]), (route, side, info)
        return
    assert not info.any(), (route, side, info)
    streaming = route in ("tile", "stream")
    for i in range(2):
        Xr = hp_householder(A[i], B[i], eps=0.0 if streaming else orc.EPS)[2]
        err = np.max(np.abs(X[i] - Xr), axis=1) / np.max(np.abs(Xr), axis=1)
        assert np.max(err) <= 1e-6, (route, side, i, np.max(err))

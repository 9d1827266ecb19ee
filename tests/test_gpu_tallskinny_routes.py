"""Every kernel route of the Gram, eigen-solver, SVD and tall-skinny QR entry points, at the shapes where the route changes.

As on the QR and least-squares paths (``test_gpu_routes.py``), kernel choice here depends on the shape alone.  The
functions below mirror the predicates of ``syrk_tn_supported`` / ``gram`` (``syrk.cu``, ``ops.cuh``),
``eigh_jacobi``, ``tsqr_local`` / ``tsqr_wide``, the completion QR of ``svd_complete_impl`` and the row chunking of
``gemm`` (``gemm.cu``), and derive every boundary from the device's ``max_smem`` and ``sm_count``.  Each case proves which
route ran with an observable that differs between the routes, without any extra ABI:

- Gram: the GEMM route is bitwise the TN GEMM that ``gram`` calls; the SYRK route makes exactly two launches and, on
  Gaussian input, differs from that GEMM.
- Eigen-solver: the one-sided route makes 4 launches, the two-sided route 3.  For n > 128 the ``JACOBI_TWO_SIDED`` option
  changes nothing (bitwise); for n <= 128 it selects the other kernel, which gives other bits on a generic matrix.
  Whether the two-sided kernel keeps the matrix in shared or in global memory has no observable: the mirror alone picks
  the last shared-memory and the first global-memory size.
- SVD: ``lq_eigh_dev`` always replays the rotation log, so ``svd``'s Vt is bitwise the transpose of its V exactly when
  ``svd`` replayed instead of taking the normalised converged columns.
- TSQR: the Householder fallback is bitwise the call made under the ``TSQR_HOUSEHOLDER`` option (both end in the blocked
  QR and the sign fix); CholeskyQR2 and BCGS2 are not.

References, with u = 2^-53 and one constant per family that is the same on every route.  Where LAPACK's result can be
held to the same bound on the same input, it is (as ``check_x`` does for least squares), which shows that the bound is
not looser than the problem:

- Gram: integer inputs in [-2^10, 2^10] make every partial sum exact, so G must equal the int64 product bitwise; on
  Gaussian input |G^ - G| <= c m u (|A|^T |A|) elementwise against an extended-precision product (float64 BLAS with twice
  the bound where that is too slow).
- Eigen-solver, against LAPACK's eigh of the same G: |lambda^_i - lambda_i|, ||G v^_i - lambda^_i v^_i|| <= c n u ||G||,
  ||V^T V - I||_max <= c n u, and sin(v^_i, v_i) <= c n u ||G|| / gap_i where that is below 0.1.
- SVD, against LAPACK's svd: |s^_i^2 - s_i^2| <= c m u s_1^2, sin(v^_i, v_i) <= c m u s_1^2 / min_j |s_i^2 - s_j^2|,
  ||A - U^ S^ V^^T||_F <= c n u ||A||_F, |U^^T U^ - I|_ij <= c m u s_1^2 / (s^_i s^_j).  ``oracle.svd_gram`` meets them too.
- TSQR: R against LAPACK (sign-fixed) to c max(m, n) u kappa, and to 1e-10 for kappa <= 1e2; residual and orthogonality
  <= 1e-12, diag(R) > 0 and tril(R) == 0 always.
"""
import numpy as np
import pytest

import linalg_b200 as lb
from oracle import linalg_oracle as orc
from test_gpu_routes import U64, _hp, conditioned, counted

REL = 1e-10
RESID = 1e-12
ORTH = 1e-12
# the constant c of each bound, the same on every route.  Measured on a B200 (1000 W): the Jacobi routes reach about 5 n u
# on eigenvalues, 73 n u on eigen-residuals (two-sided, n = 500) and 10 n u on the orthogonality of their V, whose
# rounding also sets the SVD reconstruction (7 n u); LAPACK stays below 1 n u on all of them.
C_GRAM = 2
C_EIG = 8          # eigenvalues, eigenvectors
C_EIG_RESID = 128  # ||G v - lambda v||
C_V_ORTH = 16      # ||V^T V - I|| of the Jacobi eigenvectors (eigen-solver and SVD)
C_SVD = 4          # singular values, right vectors and subspaces, U's orthogonality
C_SVD_RECON = 16   # ||A - U S V^T||_F
C_TSQR = 4

# ----------------------------------------------------------------------------- the route table
B200 = {"sm_count": 148, "max_smem": 232448}   # a B200 with 227 KB of opt-in shared memory per block
SYRK_MIN_ROWS = 16 * 64                        # syrk_tn_supported: m >= 16 * 64
SYRK_SLAB = 16                                 # rows per k-tile of syrk_tn_kernel; the rest are tail rows
ONE_SIDED_NE16_MAX = 112                       # jacobi1s_kernel<0> while ne = n padded to 16 stays below 128
ONE_SIDED_MAX = 128
EIGH_MAX_N = 2048
TWO_SIDED_STATIC_SMEM = 9216                   # the static shared memory of jacobi_kernel
CHOLQR2_ROWS_PER_COL = 4                       # tsqr_local: CholeskyQR2 for m >= 4 n (n <= 128)
BCGS2_ROWS_PER_COL = 2                         # tsqr_wide: BCGS2 for m >= 2 n (n > 128)
SINGLE_SMALL_MN = 4096                         # lq_householder_qr_dev: m * n <= 4096 on the one-CTA kernel
GEMM_ROW_CHUNK = 1 << 21                       # gemm: taller products run in row chunks


def gram_route(m, n, aligned=True):
    """gram with lda = n: the symmetric rank-k kernel when syrk_tn_supported holds, else the TN GEMM."""
    ok = 2 <= n <= 128 and n % 2 == 0 and aligned and m >= SYRK_MIN_ROWS
    return "syrk" if ok else "gemm"


def syrk_splits(m, sm_count):
    return min(sm_count, max(1, (m // SYRK_SLAB) // 4))


def two_sided_smem_bytes(n):
    ne = (n + 1) & ~1
    return (ne * (ne | 1) + 4) * 8 + (ne // 2) * 16 + 64


def eigh_route(n, max_smem):
    if not 1 <= n <= EIGH_MAX_N:
        return "refused"
    if n <= ONE_SIDED_NE16_MAX:
        return "one_sided_0"
    if n <= ONE_SIDED_MAX:
        return "one_sided_8"
    return "two_sided_smem" if two_sided_smem_bytes(n) + TWO_SIDED_STATIC_SMEM <= max_smem else "two_sided_global"


def tsqr_route(m, n):
    """The first choice of tsqr_local for well-conditioned input (a bad status word also sends it to "householder")."""
    if n <= 128:
        return "cholqr2" if m >= CHOLQR2_ROWS_PER_COL * n else "householder"
    return "bcgs2" if m >= BCGS2_ROWS_PER_COL * n else "householder"


def completion_qr_route(m, k):
    return "one_cta" if m * k <= SINGLE_SMALL_MN else "blocked"


def gemm_row_chunks(M):
    return -(-M // GEMM_ROW_CHUNK)


def last_two_sided_smem(max_smem):
    n = ONE_SIDED_MAX
    while eigh_route(n + 1, max_smem) == "two_sided_smem":
        n += 1
    return n


def full_syrk_grid_rows(sm_count):
    """Fewest rows for which the split-K SYRK grid covers every SM."""
    return 4 * SYRK_SLAB * sm_count


def check_route_table(props):
    smem, sms = props["max_smem"], props["sm_count"]
    assert eigh_route(ONE_SIDED_NE16_MAX, smem) == "one_sided_0" and eigh_route(ONE_SIDED_NE16_MAX + 1, smem) == "one_sided_8"
    assert eigh_route(ONE_SIDED_MAX, smem) == "one_sided_8"
    ns = last_two_sided_smem(smem)
    assert ns > ONE_SIDED_MAX, ("no two-sided shape fits shared memory", smem)
    assert eigh_route(ns, smem) == "two_sided_smem" and eigh_route(ns + 1, smem) == "two_sided_global", ns
    assert eigh_route(EIGH_MAX_N, smem) == "two_sided_global" and eigh_route(EIGH_MAX_N + 1, smem) == "refused"
    assert gram_route(SYRK_MIN_ROWS - 1, 128) == "gemm" and gram_route(SYRK_MIN_ROWS, 128) == "syrk"
    assert gram_route(SYRK_MIN_ROWS, 127) == "gemm" and gram_route(SYRK_MIN_ROWS, 2) == "syrk"
    assert gram_route(SYRK_MIN_ROWS, 1) == "gemm" and gram_route(SYRK_MIN_ROWS, 130) == "gemm"
    assert gram_route(SYRK_MIN_ROWS, 64, aligned=False) == "gemm"
    g = full_syrk_grid_rows(sms)
    assert syrk_splits(g - 1, sms) == sms - 1 and syrk_splits(g, sms) == sms, g
    for n in (1, 2, 17, 64, 127, 128):
        assert tsqr_route(4 * n - 1, n) == "householder" and tsqr_route(4 * n, n) == "cholqr2", n
    for n in (129, 300, 1000):
        assert tsqr_route(2 * n - 1, n) == "householder" and tsqr_route(2 * n, n) == "bcgs2", n
    assert completion_qr_route(64, 64) == "one_cta" and completion_qr_route(65, 63) == "one_cta"
    assert completion_qr_route(4096, 1) == "one_cta" and completion_qr_route(4097, 1) == "blocked"
    assert completion_qr_route(65, 65) == "blocked"
    assert gemm_row_chunks(GEMM_ROW_CHUNK) == 1 and gemm_row_chunks(GEMM_ROW_CHUNK + 37) == 2
    if (smem, sms) == (B200["max_smem"], B200["sm_count"]):
        assert ns == 166 and g == 9472


def test_route_table_boundaries_b200():
    """The mirrored predicates on a 232 448-byte, 148-SM device: eigen-solver 112 / 113 (one-sided, 16-padded / 128),
    128 / 129 (one-sided / two-sided), 166 / 167 (two-sided in shared / global memory), 2048 / 2049 (refused); SYRK from
    m = 1024 and with the full grid from m = 9472; TSQR at m = 4n (n <= 128) and m = 2n (n > 128)."""
    check_route_table(B200)


@pytest.mark.gpu
def test_route_table_boundaries_on_this_device(ctx):
    check_route_table(ctx.props())


# ----------------------------------------------------------------------------- helpers
def assert_within(label, **checks):
    """checks: name -> (error, bound).  Every error is within its bound; the message gives error / bound of each."""
    ratios = {k: float(e / b) if b > 0 else (0.0 if e == 0 else np.inf) for k, (e, b) in checks.items()}
    assert all(r <= 1.0 for r in ratios.values()), (label, ratios)


def with_option(ctx, name, fn, *args):
    ctx.set_option(name, True)
    try:
        return fn(*args)
    finally:
        ctx.set_option(name, False)


def vec_dist(a, b):
    """min ||a -+ b|| per column: 2 sin(angle / 2) for unit vectors, without the cancellation of sqrt(1 - cos^2)."""
    return np.minimum(np.linalg.norm(a - b, axis=0), np.linalg.norm(a + b, axis=0))


def isolated_gaps(vals):
    """min_{j != i} |vals_i - vals_j| (inf for a single value)."""
    d = np.abs(vals[:, None] - vals[None, :])
    np.fill_diagonal(d, np.inf)
    return d.min(axis=1)


# ----------------------------------------------------------------------------- Gram matrix
def _gram_shapes():
    return [(1023, 128), (1024, 128), (1024 + 15, 128), (2047, 64), ("grid-1", 64), ("grid", 64), ("grid+13", 128),
            (4096, 127), (4096, 1), (1024, 2), (1031, 2), (2000, 130), ((1 << 17) + 9, 32), (3000, 64, "misaligned")]


def _resolve_gram(shape, sms):
    m, n, *rest = shape
    if isinstance(m, str):
        g = full_syrk_grid_rows(sms)
        m = g - 1 if m == "grid-1" else (g if m == "grid" else g + 13)
    return m, n, bool(rest)


def _gram_id(shape):
    return "x".join(map(str, shape))


@pytest.mark.gpu
@pytest.mark.parametrize("shape", _gram_shapes(), ids=_gram_id)
def test_gram_routes(ctx, shape):
    """lq_gram_dev on both sides of m = 1024, of the full split-K grid (m = 64 sm_count), with m % 16 tail rows, odd n,
    n = 1, 2 and 130, and a base address that is 8 but not 16-byte aligned.  Integer input: bitwise the exact product on
    every route.  Gaussian input: the route's observable, and the elementwise bound."""
    m, n, misaligned = _resolve_gram(shape, ctx.props()["sm_count"])
    route = gram_route(m, n, aligned=not misaligned)
    rng = np.random.default_rng(m * 131 + n)
    off = 1 if misaligned else 0

    def run(A):
        buf = np.zeros(m * n + off)
        buf[off:] = A.ravel()
        dA, dG, dH = ctx.upload(buf), ctx.alloc(8 * n * n), ctx.alloc(8 * n * n)
        p = dA.ptr + 8 * off
        _, nl = counted(ctx, ctx.call, "lq_gram_dev", p, m, n, dG.ptr)
        ctx.call("lq_gemm_dev", 1, 0, n, n, m, 1.0, p, n, p, n, 0.0, dH.ptr, n)   # the call gram makes
        return ctx.download(dG, (n, n)), ctx.download(dH, (n, n)), nl

    Ai = rng.integers(-1024, 1025, size=(m, n)).astype(np.float64)
    G, H, nl = run(Ai)
    Ai64 = Ai.astype(np.int64)
    exact = (Ai64.T @ Ai64).astype(np.float64)
    assert np.array_equal(G, exact) and np.array_equal(H, exact), (route, m, n)

    A = rng.standard_normal((m, n))
    G, H, nl = run(A)
    if route == "gemm":
        assert np.array_equal(G, H), (m, n, "the mirror says GEMM, the result is not the GEMM's")
    else:
        assert nl == 2 and not np.array_equal(G, H), (m, n, nl, "the mirror says SYRK")
        assert np.array_equal(G, G.T)
    absA = np.abs(A)
    bound = C_GRAM * m * U64 * (absA.T @ absA)
    if m * n * n <= (1 << 25):
        Ah = _hp(A)
        err = np.abs(_hp(G) - Ah.T @ Ah).astype(np.float64)
    else:
        err, bound = np.abs(G - A.T @ A), 2 * bound
    assert_within(f"gram {m}x{n} {route}", elementwise=(np.max(err / bound), 1.0))


# ----------------------------------------------------------------------------- eigen-solver
EIG_SIZES = [1, 2, 15, 16, 17, 112, 113, 127, 128, 129, "smem_last", "global_first", 500]
EIG_KINDS = ["gram", "zero", "scalar", "diagonal", "rank_deficient", "near_equal", "graded", "indefinite"]


def _resolve_n(n, smem):
    if n == "smem_last":
        return last_two_sided_smem(smem)
    if n == "global_first":
        return last_two_sided_smem(smem) + 1
    return n


def eig_matrix(kind, n, rng):
    if kind == "gram":
        M = rng.standard_normal((n + 7, n))
        return M.T @ M
    if kind == "zero":
        return np.zeros((n, n))
    if kind == "scalar":
        return 3.0 * np.eye(n)
    if kind == "diagonal":
        return np.diag(rng.uniform(-2.0, 5.0, n))
    lam = {"rank_deficient": np.r_[rng.uniform(1.0, 2.0, n - n // 2), np.zeros(n // 2)],
           "near_equal": np.r_[1 + 1e-10, 1 - 1e-10, np.linspace(2.0, 3.0, max(n - 2, 0))][:n],
           "graded": np.logspace(0, -16, n),
           "indefinite": np.linspace(1.0, 2.0, n) * (-1.0) ** np.arange(n)}[kind]
    Q = np.linalg.qr(rng.standard_normal((n, n)))[0]
    G = (Q * lam) @ Q.T
    return (G + G.T) / 2


def eig_errors(G, lam, V, lam_ref, V_ref):
    """(error, bound) of each eigen-solver check; lam descending, lam_ref ascending (LAPACK)."""
    n = len(lam)
    lr, Vr = lam_ref[::-1], V_ref[:, ::-1]
    normG = np.max(np.abs(lr))
    scale = C_EIG * n * U64 * normG
    out = {"lambda": (np.max(np.abs(lam - lr)), scale),
           "residual": (np.max(np.linalg.norm(G @ V - V * lam, axis=0)), C_EIG_RESID * n * U64 * normG),
           "orth": (np.max(np.abs(V.T @ V - np.eye(n))), C_V_ORTH * n * U64)}
    gaps = isolated_gaps(lr)
    bound = np.divide(scale, gaps, out=np.full(n, np.inf), where=(gaps > 0) & (gaps < np.inf))
    iso = (bound < 0.1) & (scale > 0)
    if iso.any():
        out["vector"] = (np.max(vec_dist(V[:, iso], Vr[:, iso]) / bound[iso]), 1.0)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("kind", EIG_KINDS)
@pytest.mark.parametrize("n", EIG_SIZES)
def test_eigh_routes(ctx, n, kind):
    """lq_eigh_dev at every route boundary, on Gram, zero, alpha I, diagonal, rank-deficient PSD, near-equal (1 +- 1e-10),
    graded (down to 1e-16 lambda_max) and indefinite (distinct |lambda|) matrices.  The JACOBI_TWO_SIDED result meets the
    same bounds: for n <= 128 that is the two-sided kernel in shared memory."""
    smem = ctx.props()["max_smem"]
    n = _resolve_n(n, smem)
    route = eigh_route(n, smem)
    if kind == "near_equal" and n < 2:
        pytest.skip("needs two eigenvalues")
    G = eig_matrix(kind, n, np.random.default_rng(1000 * n + EIG_KINDS.index(kind)))
    dG = ctx.upload(G)

    def eigh():
        dl, dV = ctx.alloc(8 * n), ctx.alloc(8 * n * n)
        _, nl = counted(ctx, ctx.call, "lq_eigh_dev", dG.ptr, n, dl.ptr, dV.ptr)
        return ctx.download(dl, (n,)), ctx.download(dV, (n, n)), nl

    lam, V, nl = eigh()
    lam2, V2, nl2 = with_option(ctx, "JACOBI_TWO_SIDED", eigh)
    assert nl == (4 if route.startswith("one_sided") else 3), (n, route, nl)
    assert nl2 == 3, (n, nl2)
    same = np.array_equal(lam, lam2) and np.array_equal(V, V2)
    if route.startswith("two_sided"):
        assert same, (n, route, "the option must not change the n > 128 route")
    elif kind == "gram" and n >= 15:
        assert not same, (n, route, "the mirror says one-sided, the result is the two-sided kernel's")
    lam_ref, V_ref = np.linalg.eigh(G)
    assert np.all(np.diff(lam) <= 0)
    assert_within(f"lapack {kind} n={n}", **eig_errors(G, lam_ref[::-1], V_ref[:, ::-1], lam_ref, V_ref))
    assert_within(f"{route} {kind} n={n}", **eig_errors(G, lam, V, lam_ref, V_ref))
    assert_within(f"two-sided {kind} n={n}", **eig_errors(G, lam2, V2, lam_ref, V_ref))


@pytest.mark.gpu
def test_eigh_refuses_more_than_2048(ctx):
    """n = 2049: lq_eigh_dev refuses the shape (LQ_ERR_SHAPE -> ValueError) before launching anything; svd of an
    m x 2049 matrix gets LQ_ERR_UNSUPPORTED from the eigen-solver (-> NotImplementedError).  n = 2048, the documented
    maximum, is not run here: one CTA does about n^3 work per sweep, estimated (not measured) at over ten minutes."""
    n = EIGH_MAX_N + 1
    dG, dl, dV = ctx.alloc(8 * n * n), ctx.alloc(8 * n), ctx.alloc(8 * n * n)
    l0 = ctx.launches()
    with pytest.raises(ValueError):
        ctx.call("lq_eigh_dev", dG.ptr, n, dl.ptr, dV.ptr)
    assert ctx.launches() == l0
    with pytest.raises(NotImplementedError):
        lb.svd(np.random.default_rng(5).standard_normal((n + 3, n)), ctx=ctx)


# ----------------------------------------------------------------------------- SVD
SVD_SHAPES = [(3000, 64), (6000, 128), (1500, 200)]
SVD_SPECTRA = ["gaussian", "kappa1e2", "kappa1e4", "kappa1e6", "cluster", "scale1e-9", "scale1e7"]


def svd_input(spectrum, m, n, rng):
    """(A, number of leading equal singular values or 0)."""
    if spectrum.startswith("kappa"):
        return conditioned(rng, m, n, float(spectrum[5:])), 0
    if spectrum.startswith("ratio"):           # singular values from 1 down to sigma_min / sigma_max = ratio
        Um, _ = np.linalg.qr(rng.standard_normal((m, n)))
        V, _ = np.linalg.qr(rng.standard_normal((n, n)))
        return (Um * np.linspace(1.0, float(spectrum[5:]), n)) @ V.T, 0
    if spectrum == "cluster":
        k = n // 4
        Um, _ = np.linalg.qr(rng.standard_normal((m, n)))
        V, _ = np.linalg.qr(rng.standard_normal((n, n)))
        return (Um * np.r_[np.ones(k), np.logspace(-0.5, -2, n - k)]) @ V.T, k
    scale = float(spectrum[5:]) if spectrum.startswith("scale") else 1.0
    return scale * rng.standard_normal((m, n)), 0


def svd_errors(A, U, s, Vt, sigma, V_ref, cluster=0, r=None):
    """(error, bound) of each SVD check against LAPACK's sigma (descending) and V; the first r columns of U only."""
    m, n = A.shape
    r = n if r is None else r
    V = Vt.T
    s1sq = sigma[0] ** 2
    sb = C_SVD * m * U64 * s1sq
    out = {"s2": (np.max(np.abs(s ** 2 - sigma ** 2)), sb)}
    gaps = isolated_gaps(sigma ** 2)
    bound = np.divide(sb, gaps, out=np.full(n, np.inf), where=gaps > 0)
    iso = bound < 0.1
    iso[:cluster] = False
    if iso.any():
        out["vector"] = (np.max(vec_dist(V[:, iso], V_ref[:, iso]) / bound[iso]), 1.0)
    if cluster:
        P = V[:, :cluster] @ V[:, :cluster].T - V_ref[:, :cluster] @ V_ref[:, :cluster].T
        out["subspace"] = (np.linalg.norm(P, 2), sb / (sigma[cluster - 1] ** 2 - sigma[cluster] ** 2))
    Ur, sr = U[:, :r], s[:r]
    if r == n:
        out["reconstruction"] = (np.linalg.norm(A - (U * s) @ Vt), C_SVD_RECON * n * U64 * np.linalg.norm(A))
    else:
        out["columns"] = (np.linalg.norm(A @ V[:, :r] - Ur * sr), C_SVD_RECON * n * U64 * np.linalg.norm(A))
    orth = np.abs(Ur.T @ Ur - np.eye(r)) / (C_SVD * m * U64 * s1sq / np.outer(sr, sr))
    out["u_orth"] = (np.max(orth), 1.0)
    out["v_orth"] = (np.max(np.abs(Vt @ V - np.eye(n))), C_V_ORTH * n * U64)
    return out


def replay_vt(ctx, A):
    """Vt and s as the always-replaying lq_eigh_dev gives them for A^T A (formed by lq_gram_dev, as svd does)."""
    m, n = A.shape
    dA, dG, dl, dV = ctx.upload(A), ctx.alloc(8 * n * n), ctx.alloc(8 * n), ctx.alloc(8 * n * n)
    ctx.call("lq_gram_dev", dA.ptr, m, n, dG.ptr)
    ctx.call("lq_eigh_dev", dG.ptr, n, dl.ptr, dV.ptr)
    return ctx.download(dV, (n, n)).T, np.sqrt(np.maximum(ctx.download(dl, (n,)), 0.0))


def svd_route(n, sigma):
    """Direct eigenvectors when the one-sided solver ran on a PSD matrix with lambda_min > 1e-2 lambda_max."""
    return "direct" if n <= ONE_SIDED_MAX and (sigma[-1] / sigma[0]) ** 2 > 1e-2 else "replay"


def check_svd(ctx, A, cluster=0, label=""):
    m, n = A.shape
    U, s, Vt = lb.svd(A, ctx=ctx)
    _, sigma, VtL = np.linalg.svd(A, full_matrices=False)
    route = svd_route(n, sigma)
    Vr, sr = replay_vt(ctx, A)
    replayed = np.array_equal(Vt, Vr)
    assert replayed == (route == "replay"), (label, route)
    if replayed:
        assert np.array_equal(s, sr), label
    assert np.all(np.diff(s) <= 0)
    Uo, so, Vto = orc.svd_gram(A)
    assert_within(f"oracle {label}", **svd_errors(A, Uo, so, Vto, sigma, VtL.T, cluster))
    assert_within(f"{route} {label}", **svd_errors(A, U, s, Vt, sigma, VtL.T, cluster))
    return U, s, Vt


@pytest.mark.gpu
@pytest.mark.parametrize("spectrum", SVD_SPECTRA)
@pytest.mark.parametrize("shape", SVD_SHAPES, ids=_gram_id)
def test_svd_spectra(ctx, shape, spectrum):
    """Gaussian, geometric kappa = 1e2, 1e4, 1e6 (where the A^T A route is weakest), a block of equal singular values
    (subspace checks only) and scaled input, on the one-sided (direct and replayed eigenvectors) and two-sided routes."""
    m, n = shape
    A, cluster = svd_input(spectrum, m, n, np.random.default_rng(m + n + SVD_SPECTRA.index(spectrum)))
    check_svd(ctx, A, cluster, f"{spectrum} {m}x{n}")


@pytest.mark.gpu
@pytest.mark.parametrize("ratio,route", [(0.12, "direct"), (0.08, "replay")])
@pytest.mark.parametrize("n", [64, 128])
def test_svd_direct_replay_cut(ctx, n, ratio, route):
    """sigma_min / sigma_max = 0.12 takes the normalised converged columns (lambda ratio 0.0144 > 1e-2), 0.08 replays."""
    A, _ = svd_input(f"ratio{ratio}", 4000, n, np.random.default_rng(n))
    assert svd_route(n, np.linalg.svd(A, compute_uv=False)) == route
    check_svd(ctx, A, 0, f"cut {ratio} n={n}")


@pytest.mark.gpu
def test_svd_gemm_row_chunks(ctx):
    """2^21 + 37 rows: U = A V S^-1 runs as two row chunks of the GEMM."""
    m, n = GEMM_ROW_CHUNK + 37, 24
    assert gemm_row_chunks(m) == 2
    check_svd(ctx, np.random.default_rng(21).standard_normal((m, n)), 0, "row chunks")


@pytest.mark.gpu
def test_svd_wide_is_the_transposed_call(ctx):
    A = np.random.default_rng(8).standard_normal((700, 40))
    U, s, Vt = lb.svd(A, ctx=ctx)
    U2, s2, Vt2 = lb.svd(np.ascontiguousarray(A.T), ctx=ctx)
    assert np.array_equal(U2, Vt.T) and np.array_equal(s2, s) and np.array_equal(Vt2, U.T)


@pytest.mark.gpu
def test_svd_tol_cuts_small_singular_values(ctx):
    """tol = 1e-3 on a geometric spectrum from 1 to 1e-6: rank = #(sigma > tol), no sigma lies within the bound of tol.  s
    keeps the small values, U's first r columns are A V_r / s_r, the rest come from the completion (orthonormal, and
    orthogonal to U_r to within U_r's own bound)."""
    m, n, tol = 2000, 40, 1e-3
    A = conditioned(np.random.default_rng(40), m, n, 1e6)
    _, sigma, VtL = np.linalg.svd(A, full_matrices=False)
    r = int(np.sum(sigma > tol))
    margin = C_SVD * m * U64 * sigma[0] ** 2 / tol     # |s^ - sigma| near tol is at most about this
    assert 0 < r < n and margin < np.min(np.abs(sigma - tol))
    U, s, Vt = lb.svd(A, tol, ctx=ctx, seed=7)
    assert int(np.sum(s > tol)) == r
    assert_within("tol", **svd_errors(A, U, s, Vt, sigma, VtL.T, r=r))
    Uo, so, Vto = orc.svd_gram(A, tol, rng=np.random.RandomState(7))
    assert_within("oracle tol", **svd_errors(A, Uo, so, Vto, sigma, VtL.T, r=r))
    assert np.linalg.norm(A @ Vt[r] / s[r] - U[:, r]) > 0.1     # column r is the completion's, not A v_r / s_r
    Uc = U[:, r:]
    assert np.max(np.abs(Uc.T @ Uc - np.eye(n - r))) <= ORTH
    assert np.max(np.abs(U[:, :r].T @ Uc)) <= C_SVD * m * U64 * (sigma[0] / s[r - 1]) ** 2


# ----------------------------------------------------------------------------- SVD completion
# (m, n, rank): rank-deficient by exactly zero columns, so that the eigen-solver sees exact zeros
COMPLETION_CASES = [(64, 64, 0), (65, 65, 0), (100, 40, 0), (103, 40, 0), (65, 64, 1), (66, 64, 1), (4096, 2, 1),
                    (4097, 2, 1), (4096, 8, 7), (4097, 8, 7)]


@pytest.mark.gpu
@pytest.mark.parametrize("m,n,rank", COMPLETION_CASES)
def test_svd_completion_routes(ctx, m, n, rank):
    """The completion's QR of m x (n - rank) candidates on both sides of m (n - rank) = 4096, with rank 0 (zero matrix,
    square and not), 1 and n - 1.  From the global np.random: U's completed columns equal the oracle's (the reference's
    algorithm, same draws) up to a per-column sign.  With seed=: U orthonormal with its completion, reconstruction."""
    k = n - rank
    route = completion_qr_route(m, k)
    dZ, dQ, dR = ctx.upload(np.random.default_rng(k).standard_normal((m, k))), ctx.alloc(8 * m * k), ctx.alloc(8 * k * k)
    _, nl = counted(ctx, ctx.call, "lq_householder_qr_dev", dZ.ptr, m, k, dQ.ptr, dR.ptr)
    assert (nl == 1) == (route == "one_cta"), (m, k, route, nl)
    A = np.random.default_rng(m * n + rank).standard_normal((m, n))
    A[:, rank:] = 0.0
    np.random.seed(rank + 3)
    U, s, Vt = lb.svd(A, ctx=ctx)
    Uo, so, _ = orc.svd_gram(A, rng=np.random.RandomState(rank + 3))
    assert int(np.sum(s > 1e-12)) == rank == int(np.sum(so > 1e-12))
    sg = np.sign(np.sum(U[:, rank:] * Uo[:, rank:], axis=0))
    assert orc.rel_max_err(U[:, rank:] * sg, Uo[:, rank:]) <= REL
    U2, s2, Vt2 = lb.svd(A, ctx=ctx, seed=11)
    assert np.array_equal(s2, s)
    assert np.max(np.abs(U2.T @ U2 - np.eye(n))) <= ORTH
    assert np.linalg.norm(A - (U2 * s2) @ Vt2) <= C_SVD_RECON * n * U64 * np.linalg.norm(A)


# ----------------------------------------------------------------------------- TSQR
def tsqr_input(kind, m, n, rng):
    """(A, route forced by the data or None, whether R is unique)."""
    if kind.startswith("kappa"):
        kappa = float(kind[5:])
        return conditioned(rng, m, n, kappa), ("householder" if kappa ** 2 >= 1e10 else None), True
    A = rng.standard_normal((m, n))
    if kind == "zero_col":          # Cholesky breakdown (n <= 128) / a bad panel status (n > 128: column 150)
        A[:, min(n - 1, 150) if n > 128 else n // 2] = 0.0
        return A, "householder", False
    if kind == "dependent":
        A[:, n // 2] = A[:, 1] + 2.0 * A[:, 2]
        return A, "householder", False
    if kind == "near_dependent_panel":   # second panel = first panel x M + 1e-8 noise: kappa about 1e8
        A[:, 128:] = A[:, :128] @ (rng.standard_normal((128, n - 128)) / np.sqrt(128)) + 1e-8 * rng.standard_normal((m, n - 128))
        return A, None, True
    if kind == "combination_panel":      # a column of the second panel is a combination of the first panel's
        A[:, 140] = A[:, 3] + 2.0 * A[:, 5]
        return A, None, False
    return A, None, True


TSQR_CASES = ([(4 * n + d, n, "normal") for n in (1, 2, 17, 64, 127, 128) for d in (-1, 0)]
              + [(1023, 128, "normal"), (1024, 128, "normal"), (2005, 33, "normal"), (1029, 127, "normal")]
              + [(1, 1, "normal"), (2, 2, "normal"), (5, 3, "normal"), (31, 31, "normal"), (33, 32, "normal"), (64, 64, "normal")]
              + [(GEMM_ROW_CHUNK + 37, 24, "normal")]
              + [(4000, 40, "kappa1e3"), (4000, 40, "kappa1e7"), (3000, 50, "zero_col"), (3000, 50, "dependent")]
              + [(1000, 129, "normal"), (1000, 130, "normal"), (1000, 131, "normal"), (2000, 256, "normal"), (1500, 300, "normal")]
              + [(5000, 1000, "normal"), (257, 129, "normal"), (258, 129, "normal"), (599, 300, "normal"), (600, 300, "normal")]
              + [(1200, 200, "zero_col"), (1200, 256, "near_dependent_panel"), (1200, 256, "combination_panel")])


@pytest.mark.gpu
@pytest.mark.parametrize("m,n,kind", TSQR_CASES, ids=[f"{m}x{n}_{k}" for m, n, k in TSQR_CASES])
def test_tsqr_routes(ctx, m, n, kind):
    """lb.tsqr at m = 4n - 1 / 4n (n <= 128) and 2n - 1 / 2n (n > 128), the SYRK boundary inside CholeskyQR2, odd n and
    m % 16 != 0, tiny shapes on the blocked QR (fewer rows than its 32-column panel), a 1-column last BCGS2 panel, 2^21 + 37
    rows (GEMM row chunks), the reference's 5000 x 1000, and the data-driven fallbacks (kappa^2 >= 1e10, a zero column, a
    dependent column).  The device entry gives the same bits."""
    A, forced_route, unique = tsqr_input(kind, m, n, np.random.default_rng(m * 7 + n))
    route = forced_route or tsqr_route(m, n)
    Q, R = lb.tsqr(A, ctx=ctx)
    Qh, Rh = with_option(ctx, "TSQR_HOUSEHOLDER", lb.tsqr, A)
    same = np.array_equal(Q, Qh) and np.array_equal(R, Rh)
    if kind in ("near_dependent_panel", "combination_panel"):
        route = "householder" if same else "bcgs2"
    assert same == (route == "householder"), (m, n, kind, route)
    dA, dQ, dR = ctx.upload(A), ctx.alloc(8 * m * n), ctx.alloc(8 * n * n)
    ctx.call("lq_tsqr_dev", dA.ptr, m, n, dQ.ptr, dR.ptr)
    assert np.array_equal(ctx.download(dQ, (m, n)), Q) and np.array_equal(ctx.download(dR, (n, n)), R)
    assert np.all(np.tril(R, -1) == 0.0)
    assert np.all(np.diag(R) > 0) if unique else np.all(np.diag(R) >= 0)
    assert orc.qr_residual(A, Q, R) <= RESID and orc.orth_error(Q) <= ORTH, (m, n, kind, route)
    if unique:
        _, Ro = orc.tsqr_reference(A)
        sv = np.linalg.svd(A, compute_uv=False)
        kappa = sv[0] / sv[-1]
        err = orc.rel_max_err(R, Ro)
        assert_within(f"tsqr {m}x{n} {kind} {route}", R=(err, C_TSQR * max(m, n) * U64 * kappa))
        if kappa <= 1e2:
            assert err <= REL, (m, n, kind, err)

"""Every route on NaN / +-Inf input and on pre-filled outputs.

Pool memory from an earlier call usually holds the finite values a kernel would write again, and several kernels share
hardware between matrices (four 32 x 32 matrices per warp in the batched Householder QR, two in the batched MGS, four
warps per CTA in the batched SVD, right-hand sides in the DMMA tiles of the least-squares tile kernel).  With finite data
an unwritten output element or a structural zero times another matrix's value goes unnoticed; with NaN it does not
(0 * NaN = NaN).  So, one representative shape per route from the route tables of ``test_gpu_routes.py``,
``test_gpu_tallskinny_routes.py`` and ``test_gpu_scaling.py`` (the QR, least-squares and GEMM routes held by their launch
counts):

1. every output element is written: outputs pre-filled with NaN (integers 0x7fffffff) and with a finite sentinel (integers
   -7) give the same bits;
2. batch containment: one non-finite entry in matrix i leaves every other matrix's outputs bitwise those of the clean
   batch, with i sharing a warp / CTA with clean matrices;
3. right-hand-side containment: NaN in column k of B leaves every other column of X bitwise unchanged, column k non-finite;
4. decisions: the QR and least-squares routes raise exactly when the oracle does (never, for these inputs) and return
   non-finite R / X whenever the oracle's are; svd, svd_batched and the eigen-solver raise nothing and return NaN in s /
   lambda (the eigen-solvers treat any non-finite G as unresolvable: every eigenvalue NaN, V = I); non-finite calls are
   bitwise deterministic, NaN payloads included;
5. the CholeskyQR2 verdict declines non-finite input and a Gram matrix that overflows: bitwise the TSQR_HOUSEHOLDER result;
6. GEMM with beta = 0 does not read C.

Non-finite positions: the first entry, one interior entry, the last entry; values NaN, +Inf, -Inf.
"""
import ctypes as C
import itertools

import numpy as np
import pytest

import linalg_b200 as lb
from oracle import linalg_oracle as orc
from test_gpu_routes import assert_route, counted, hh_qr_route, lstsq_route, mgs_qr_route
from test_gpu_scaling import GEMM_CASES, gemm_route
from test_gpu_tallskinny_routes import eigh_route, gram_route, tsqr_route, with_option

pytestmark = pytest.mark.gpu

VALUES = {"nan": np.nan, "inf": np.inf, "-inf": -np.inf}
POSITIONS = ("first", "interior", "last")
INT_FILL = {"nan": 0x7FFFFFFF, "finite": -7}
FLOAT_FILL = {"nan": np.nan, "finite": -7.0}


def poke(A, pos, value):
    """A copy of the 2-D A with `value` at its first, an interior or its last entry."""
    A = A.copy()
    m, n = A.shape
    A[{"first": (0, 0), "interior": (m // 2, n // 2), "last": (m - 1, n - 1)}[pos]] = value
    return A


def bits(x):
    return np.ascontiguousarray(x).view(np.uint64 if x.dtype == np.float64 else np.uint32)


def same_bits(label, a, b):
    assert a.shape == b.shape and np.array_equal(bits(a), bits(b)), label


def combos():
    return list(itertools.product(VALUES, POSITIONS))


# ----------------------------------------------------------------------------- device calls with pre-filled outputs
class Dev:
    """One device entry point: `ins` (name -> array) are uploaded, `outs` (name -> (shape, dtype)) are allocated and
    pre-filled, `args` lists the call's arguments after ctx (a str names a buffer, anything else is passed as is)."""

    def __init__(self, name, ins, outs, args, route=None, matrices=1):
        self.name, self.ins, self.outs, self.args, self.route, self.matrices = name, ins, outs, args, route, matrices

    def run(self, ctx, fill="nan"):
        bufs = {k: ctx.upload(v) for k, v in self.ins.items()}
        for k, (shape, dt) in self.outs.items():
            bufs[k] = ctx.upload(np.full(shape, (INT_FILL if dt == np.int32 else FLOAT_FILL)[fill], dtype=dt))
        args = [bufs[a].ptr if isinstance(a, str) else a for a in self.args]
        _, nl = counted(ctx, ctx.call, self.name, *args)
        if self.route is not None:
            assert_route(self.route, nl, self.matrices)
        return {k: ctx.download(bufs[k], shape, dtype=dt) for k, (shape, dt) in self.outs.items()}


def f64(*shape):
    return (shape, np.float64)


def i32(*shape):
    return (shape, np.int32)


def hh_qr_batched(A, route):
    b, m, n = A.shape
    return Dev("lq_householder_qr_batched_dev", {"A": A}, {"Q": f64(b, m, n), "R": f64(b, n, n)},
               ["A", b, m, n, "Q", "R", 0], route, b)


def hh_qr_single(A, route):
    m, n = A.shape
    return Dev("lq_householder_qr_dev", {"A": A}, {"Q": f64(m, n), "R": f64(n, n)}, ["A", m, n, "Q", "R"], route, 1)


def mgs_qr_batched(A, route):
    b, m, n = A.shape
    return Dev("lq_mgs_qr_batched_dev", {"A": A}, {"Q": f64(b, m, n), "R": f64(b, n, n), "info": i32(b)},
               ["A", b, m, n, 0, "Q", "R", "info"], route, b)


def mgs_qr_single(A, route):
    m, n = A.shape
    return Dev("lq_mgs_qr_dev", {"A": A}, {"Q": f64(m, n), "R": f64(n, n), "info": i32(1)},
               ["A", m, n, 0, "Q", "R", "info"], route, 1)


LS_DEV = {"hh": "lq_lstsq_householder_batched_info_dev", "mgs": "lq_lstsq_mgs_batched_dev"}


def lstsq(method, A, B, route):
    b, m, n = A.shape
    k = B.shape[2]
    return Dev(LS_DEV[method], {"A": A, "B": B}, {"X": f64(b, n, k), "info": i32(b)},
               ["A", "B", b, m, n, k, "X", "info"], route, b)


def svd_batched_dev(A):
    b, m, n = A.shape
    return Dev("lq_svd_gram_batched_dev", {"A": A}, {"U": f64(b, m, n), "s": f64(b, n), "Vt": f64(b, n, n), "rank": i32(b)},
               ["A", b, m, n, 1e-12, "U", "s", "Vt", "rank"])


def eigh_dev(G):
    n = G.shape[0]
    return Dev("lq_eigh_dev", {"G": G}, {"lam": f64(n), "V": f64(n, n)}, ["G", n, "lam", "V"])


def tsqr_dev(A):
    m, n = A.shape
    return Dev("lq_tsqr_dev", {"A": A}, {"Q": f64(m, n), "R": f64(n, n)}, ["A", m, n, "Q", "R"])


def lstsq_tsqr_dev(A, B):
    (m, n), k = A.shape, B.shape[1]
    return Dev("lq_lstsq_tsqr_dev", {"A": A, "B": B}, {"X": f64(n, k), "info": i32(1)}, ["A", m, n, "B", k, "X", "info"])


def run_svd_gram_dev(ctx, A, fill):
    """lq_svd_gram_dev (its rank is a host pointer): U, s, Vt pre-filled, rank pre-set."""
    m, n = A.shape
    dA = ctx.upload(A)
    dU, ds, dV = (ctx.upload(np.full(s, FLOAT_FILL[fill])) for s in ((m, n), (n,), (n, n)))
    rank = C.c_int(INT_FILL[fill])
    ctx.call("lq_svd_gram_dev", dA.ptr, m, n, 1e-12, dU.ptr, ds.ptr, dV.ptr, C.byref(rank))
    return {"U": ctx.download(dU, (m, n)), "s": ctx.download(ds, (n,)), "Vt": ctx.download(dV, (n, n)),
            "rank": np.array([rank.value], np.int32)}


# ----------------------------------------------------------------------------- representative shapes of every route
def gauss(shape, *key):
    return np.random.default_rng(sum(shape) * 7919 + len(key)).standard_normal(shape)


def write_cases(smem):
    """(label, Dev) with Gaussian input for every route of every device entry point."""
    out = []
    for label, (b, m, n) in (("hh_small", (9, 40, 24)), ("hh_qr32", (9, 32, 32)), ("hh_blocked_batched", (2, 169, 169))):
        out.append((label, hh_qr_batched(gauss((b, m, n)), hh_qr_route(m, n, smem, True))))
    for label, (m, n) in (("hh_single_one_cta", (64, 64)), ("hh_single_blocked", (255, 200))):
        out.append((label, hh_qr_single(gauss((m, n)), hh_qr_route(m, n, smem, False))))
    for label, (b, m, n) in (("mgs_small", (9, 40, 24)), ("mgs_qr32", (9, 32, 32)), ("mgs_large", (2, 121, 121))):
        out.append((label, mgs_qr_batched(gauss((b, m, n)), mgs_qr_route(m, n, smem))))
    for label, (m, n) in (("mgs_single_small", (40, 24)), ("mgs_single_large", (121, 121))):
        out.append((label, mgs_qr_single(gauss((m, n)), mgs_qr_route(m, n, smem))))
    for method, shape in LS_ROUTES:
        b, (m, n, k) = (9 if shape[0] <= 1000 and shape[1] <= 64 else 2), shape
        route = lstsq_route(method, m, n, k, smem)
        out.append((f"ls_{method}_{route}", lstsq(method, gauss((b, m, n)), gauss((b, m, k), 1), route)))
    out.append(("svd_batched_kernel", svd_batched_dev(gauss((9, 256, 16)))))
    out.append(("svd_batched_per_matrix", svd_batched_dev(gauss((2, 40, 33)))))
    for n in EIG_NS:
        M = gauss((n + 7, n))
        out.append((f"eigh_{eigh_route(n, smem)}", eigh_dev(M.T @ M)))
    for m, n in GRAM_SHAPES:
        out.append((f"gram_{gram_route(m, n)}", Dev("lq_gram_dev", {"A": gauss((m, n))}, {"G": f64(n, n)}, ["A", m, n, "G"])))
    for m, n in TSQR_SHAPES:
        out.append((f"tsqr_{tsqr_route(m, n)}", tsqr_dev(gauss((m, n)))))
    for label, (m, n, k) in LSTSQ_TSQR_SHAPES:
        out.append((f"lstsq_tsqr_{label}", lstsq_tsqr_dev(gauss((m, n)), gauss((m, k), 1))))
    return out


LS_ROUTES = [("hh", (100, 20, 4)), ("hh", (1000, 64, 32)), ("hh", (120, 64, 33)), ("hh", (700, 300, 3)),
             ("mgs", (100, 20, 4)), ("mgs", (120, 64, 33)), ("mgs", (700, 300, 3))]
EIG_NS = [64, 150, 200]                   # one-sided, two-sided in shared memory, two-sided in global memory
GRAM_SHAPES = [(2048, 64), (1023, 128)]   # SYRK, GEMM
TSQR_SHAPES = [(4000, 40), (1000, 130), (100, 40)]   # CholeskyQR2, BCGS2 panels, Householder
# strip: [G2 | C] in the SYRK strip kernel (odd nrhs padded with a zero column); plain: SYRK / GEMM and a TN GEMM
LSTSQ_TSQR_SHAPES = [("strip_even", (4096, 64, 4)), ("strip_odd", (4096, 64, 5)), ("plain", (1000, 32, 6)),
                     ("householder", (255, 64, 4))]
SVD_SHAPES = [(3000, 64), (1500, 200)]    # one-sided, two-sided eigen-solver


@pytest.fixture(scope="module")
def smem(ctx):
    return ctx.props()["max_smem"]


@pytest.fixture(scope="module")
def cases(smem):
    return dict(write_cases(smem))


WRITE_LABELS = [label for label, _ in write_cases(232448)]


# ----------------------------------------------------------------------------- 1. every output element is written
@pytest.mark.parametrize("label", WRITE_LABELS)
def test_every_output_element_is_written(ctx, cases, label):
    dev = cases[label]
    a, b = dev.run(ctx, "nan"), dev.run(ctx, "finite")
    if "info" in a and (a["info"].any() or b["info"].any()):
        same_bits(f"{label} info", a["info"], b["info"])
        return
    for k in a:
        same_bits(f"{label} {k}", a[k], b[k])


@pytest.mark.parametrize("label", ["one_sided", "two_sided"])
def test_svd_gram_every_output_element_is_written(ctx, label):
    m, n = SVD_SHAPES[0 if label == "one_sided" else 1]
    A = gauss((m, n))
    a, b = run_svd_gram_dev(ctx, A, "nan"), run_svd_gram_dev(ctx, A, "finite")
    for k in a:
        same_bits(f"svd {label} {k}", a[k], b[k])


# ----------------------------------------------------------------------------- 2. batch containment
def poisoned_batches(A, idx):
    """(i, value, position, batch with one non-finite entry in matrix i), i cycling over idx."""
    for c, (v, pos) in enumerate(combos()):
        i = idx[c % len(idx)]
        P = A.copy()
        P[i] = poke(A[i], pos, VALUES[v])
        yield i, v, pos, P


def containment_cases(smem):
    """(label, make Dev from A (and B), A, B or None, poisoned matrices): 9 matrices where the kernel packs several per
    warp / CTA; i = 0 and 7 (mod 4 = 0 and 3 for hh_qr32_c8), 5 and 2 (both halves of an mgs_qr32 warp pair), 8 (the
    ragged last group)."""
    idx9 = [0, 7, 2, 5, 8]
    out = [("hh_qr32", lambda A, B: hh_qr_batched(A, "qr32"), gauss((9, 32, 32)), None, idx9),
           ("hh_small", lambda A, B: hh_qr_batched(A, "small"), gauss((9, 40, 24)), None, idx9),
           ("hh_blocked_batched", lambda A, B: hh_qr_batched(A, "blocked"), gauss((3, 169, 169)), None, [0, 2]),
           ("mgs_qr32", lambda A, B: mgs_qr_batched(A, "qr32"), gauss((9, 32, 32)), None, idx9),
           ("mgs_small", lambda A, B: mgs_qr_batched(A, "small"), gauss((9, 40, 24)), None, idx9),
           ("mgs_large", lambda A, B: mgs_qr_batched(A, "large"), gauss((3, 121, 121)), None, [0, 2]),
           ("svd_batched_kernel", lambda A, B: svd_batched_dev(A), gauss((9, 256, 16)), None, idx9),
           ("svd_batched_per_matrix", lambda A, B: svd_batched_dev(A), gauss((3, 40, 33)), None, [0, 2])]
    for method, (m, n, k) in LS_ROUTES:
        route = lstsq_route(method, m, n, k, smem)
        b = 9 if route in ("tile", "stream") else 3
        out.append((f"ls_{method}_{route}", (lambda meth, r: lambda A, B: lstsq(meth, A, B, r))(method, route),
                    gauss((b, m, n)), gauss((b, m, k), 1), idx9 if b == 9 else [0, 2]))
    return out


CONTAIN_LABELS = [c[0] for c in containment_cases(232448)]


@pytest.mark.parametrize("label", CONTAIN_LABELS)
def test_batch_containment(ctx, smem, label):
    _, make, A, B, idx = next(c for c in containment_cases(smem) if c[0] == label)
    clean = make(A, B).run(ctx)
    for i, v, pos, P in poisoned_batches(A, idx):
        got = make(P, B).run(ctx)
        others = [j for j in range(len(A)) if j != i]
        for k in clean:
            same_bits(f"{label} matrix {i} {v} at {pos}: {k} of the others", got[k][others], clean[k][others])


# ----------------------------------------------------------------------------- 3. right-hand-side containment
def rhs_cases(smem):
    out = []
    for method, (m, n, k) in LS_ROUTES:
        if k < 2:
            continue
        route = lstsq_route(method, m, n, k, smem)
        out.append((f"ls_{method}_{route}", (lambda meth, r: lambda A, B: lstsq(meth, A[None], B[None], r))(method, route),
                    m, n, k))
    for label, (m, n, k) in LSTSQ_TSQR_SHAPES:
        out.append((f"lstsq_tsqr_{label}", lstsq_tsqr_dev, m, n, k))
    return out


RHS_LABELS = [c[0] for c in rhs_cases(232448)]


@pytest.mark.parametrize("label", RHS_LABELS)
def test_rhs_containment(ctx, smem, label):
    _, make, m, n, k = next(c for c in rhs_cases(smem) if c[0] == label)
    A, B = gauss((m, n)), gauss((m, k), 1)
    X0 = make(A, B).run(ctx)["X"].reshape(n, k)
    for col in sorted({0, k // 2, k - 1}):
        for v in VALUES:
            Bp = B.copy()
            Bp[m // 2, col] = VALUES[v]
            out = make(A, Bp).run(ctx)
            X = out["X"].reshape(n, k)
            assert not out["info"].any(), (label, col, v)
            keep = [c for c in range(k) if c != col]
            same_bits(f"{label} nan in column {col}: the other columns", X[:, keep], X0[:, keep])
            assert not np.isfinite(X[:, col]).all(), (label, col, v)


def test_rhs_containment_mgs_entry_point(ctx):
    """least_squares_qr (the host MGS entry point) on a tile shape: column k alone turns non-finite."""
    m, n, k = 100, 20, 4
    A, B = gauss((m, n)), gauss((m, k), 1)
    X0 = lb.least_squares_qr(A, B, ctx=ctx).reshape(n, k)
    for col in range(k):
        Bp = B.copy()
        Bp[0, col] = np.nan
        X = lb.least_squares_qr(A, Bp, ctx=ctx).reshape(n, k)
        keep = [c for c in range(k) if c != col]
        same_bits(f"mgs column {col}", X[:, keep], X0[:, keep])
        assert np.isnan(X[:, col]).all(), col


# ----------------------------------------------------------------------------- 4. decisions against the oracle
def outcome(fn):
    """(raised exception type or None, result)."""
    with np.errstate(all="ignore"):
        try:
            return None, fn()
        except (ValueError, np.linalg.LinAlgError) as e:
            return type(e), None


QR_DECISIONS = [("hh", "small", (40, 24), True), ("hh", "qr32", (32, 32), True), ("hh", "blocked", (169, 169), True),
                ("hh", "small", (64, 64), False), ("hh", "blocked", (255, 200), False),
                ("mgs", "small", (40, 24), True), ("mgs", "qr32", (32, 32), True), ("mgs", "large", (121, 121), True)]


@pytest.mark.parametrize("method,route,shape,batched", QR_DECISIONS,
                         ids=[f"{m}_{r}_{'batched' if b else 'single'}" for m, r, _, b in QR_DECISIONS])
def test_qr_decisions_follow_the_oracle(ctx, smem, method, route, shape, batched):
    m, n = shape
    assert (hh_qr_route(m, n, smem, batched) if method == "hh" else mgs_qr_route(m, n, smem)) == route
    A0 = gauss(shape)
    for v, pos in combos():
        A = poke(A0, pos, VALUES[v])
        if method == "hh":
            ref = outcome(lambda: orc.householder_qr(A))
            call = lambda: outcome(lambda: lb.householder_qr_batched(A[None], ctx=ctx) if batched else lb.householder_qr(A, ctx=ctx))
        else:
            ref = outcome(lambda: orc.mgs_qr(A))
            call = lambda: outcome(lambda: lb.qr_batched(A[None], ctx=ctx) if batched else lb.qr(A, ctx=ctx))
        got = call()
        assert got[0] == ref[0], (method, route, v, pos, got[0], ref[0])
        if ref[1] is not None:
            assert np.isfinite(got[1][1]).all() == np.isfinite(ref[1][1]).all(), (method, route, v, pos)
            for x, y in zip(got[1], call()[1]):
                same_bits(f"{method} {route} {v} at {pos} determinism", x, y)


@pytest.mark.parametrize("method,shape", LS_ROUTES, ids=[f"{m}_{'x'.join(map(str, s))}" for m, s in LS_ROUTES])
def test_least_squares_decisions_follow_the_oracle(ctx, smem, method, shape):
    m, n, k = shape
    route = lstsq_route(method, m, n, k, smem)
    A0, B = gauss((m, n)), gauss((m, k), 1)
    host = lb.least_squares_householder_qr_batched if method == "hh" else lb.least_squares_qr_batched
    ref_fn = orc.lstsq_householder if method == "hh" else orc.lstsq_mgs
    for v, pos in combos():
        A = poke(A0, pos, VALUES[v])
        ref = outcome(lambda: ref_fn(A, B))
        got = outcome(lambda: host(A[None], B[None], ctx=ctx))
        assert got[0] == ref[0], (method, route, v, pos, got[0], ref[0])
        if ref[1] is not None:
            assert np.isfinite(got[1]).all() == np.isfinite(ref[1]).all(), (method, route, v, pos)
            same_bits(f"{method} {route} determinism", got[1], outcome(lambda: host(A[None], B[None], ctx=ctx))[1])


def test_svd_nonfinite_input_gives_nan(ctx):
    """svd: no exception, NaN in s where the reference returns no all-finite s, for NaN / Inf at every position and for a
    finite A whose Gram matrix overflows; the same bits twice.  The eigen-solver sees a non-finite G and returns NaN for
    every eigenvalue, so rank = 0 and U is the seeded completion."""
    for m, n in SVD_SHAPES:
        A0 = gauss((m, n))
        inputs = [(f"{v} at {pos}", poke(A0, pos, VALUES[v])) for v, pos in combos()] + [("overflow", np.ldexp(A0, 520))]
        for label, A in inputs:
            U, s, Vt = lb.svd(A, ctx=ctx, seed=1)
            assert np.isnan(s).all(), (m, n, label, s[:4])
            U2, s2, Vt2 = lb.svd(A, ctx=ctx, seed=1)
            for x, y in ((U, U2), (s, s2), (Vt, Vt2)):
                same_bits(f"svd {m}x{n} {label} determinism", x, y)


def test_svd_parent_failures_are_gone(ctx):
    """NaN in one column of A (the single-matrix route): every slot of s and Vt is written (the sort is a permutation) and
    no NaN eigenvalue turns into sigma = 0."""
    m, n = SVD_SHAPES[0]
    A = poke(gauss((m, n)), "interior", np.nan)
    a, b = run_svd_gram_dev(ctx, A, "nan"), run_svd_gram_dev(ctx, A, "finite")
    for k in ("s", "Vt", "rank"):
        same_bits(f"svd nan {k}", a[k], b[k])
    assert np.isnan(a["s"]).all() and a["rank"][0] == 0 and not (a["s"] == 0).any()


def test_svd_batched_routes_agree_on_nonfinite_input(ctx):
    """svd_batched's warp-per-matrix kernel and svd (what the per-matrix route runs, bitwise) on the same matrices: no
    exception, the same rank and the same NaN entries of s; the kernel route twice gives the same bits."""
    A0 = gauss((9, 256, 16))
    batch = np.stack([poke(A0[c], pos, VALUES[v]) for c, (v, pos) in enumerate(combos())])
    U, s, Vt = lb.svd_batched(batch, ctx=ctx, seed=2)
    out = svd_batched_dev(batch).run(ctx)
    same_bits("svd_batched determinism s", out["s"], svd_batched_dev(batch).run(ctx)["s"])
    for i in range(len(batch)):
        U1, s1, Vt1 = lb.svd(batch[i], ctx=ctx, seed=2)
        assert np.isnan(s[i]).any() and np.array_equal(np.isnan(s[i]), np.isnan(s1)), i
        assert out["rank"][i] == int(np.sum(s1 > 1e-12)), i


@pytest.mark.parametrize("n", EIG_NS)
def test_eigh_nonfinite_input_gives_nan(ctx, smem, n):
    """lq_eigh_dev on G with NaN / Inf at the first, an interior and the last entry, and on an overflowed Gram matrix: every
    eigenvalue NaN, V = I (the replay of no rotation), every output written, the same bits twice."""
    M = gauss((n + 7, n))
    G0 = M.T @ M
    with np.errstate(over="ignore"):
        Gover = np.ldexp(M, 520).T @ np.ldexp(M, 520)
    for label, G in [(f"{v} at {pos}", poke(G0, pos, VALUES[v])) for v, pos in combos()] + [("overflow", Gover)]:
        dev = eigh_dev(G)
        a, b = dev.run(ctx, "nan"), dev.run(ctx, "finite")
        for k in a:
            same_bits(f"eigh {eigh_route(n, smem)} {label} {k}", a[k], b[k])
        assert np.isnan(a["lam"]).all() and np.array_equal(a["V"], np.eye(n)), (n, label)


# ----------------------------------------------------------------------------- 5. the CholeskyQR2 verdict
def tsqr_inputs(m, n):
    A0 = gauss((m, n))
    return [(f"{v} at {pos}", poke(A0, pos, VALUES[v])) for v, pos in combos()] + [("overflow", np.ldexp(A0, 520))]


@pytest.mark.parametrize("m,n", TSQR_SHAPES[:2], ids=["cholqr2", "bcgs2"])
def test_tsqr_declines_nonfinite_input(ctx, m, n):
    """lq_tsqr_dev: NaN / Inf in A or a Gram matrix that overflows (column norms 2^520) fail the CholeskyQR2 verdict (a
    NaN pivot is breakdown, a NaN or infinite cond^2 estimate is ill-conditioned); both the n <= 128 route and the BCGS2
    panels (n > 128, any failed panel) then run the blocked Householder QR, bitwise the TSQR_HOUSEHOLDER result."""
    assert tsqr_route(m, n) in ("cholqr2", "bcgs2")
    for label, A in tsqr_inputs(m, n):
        got = tsqr_dev(A).run(ctx)
        ref = with_option(ctx, "TSQR_HOUSEHOLDER", tsqr_dev(A).run, ctx)
        for k in got:
            same_bits(f"tsqr {m}x{n} {label} {k}", got[k], ref[k])


@pytest.mark.parametrize("label", ["strip_even", "strip_odd", "plain"])
def test_lstsq_tsqr_declines_nonfinite_input(ctx, label):
    m, n, k = dict(LSTSQ_TSQR_SHAPES)[label]
    B = gauss((m, k), 1)
    for lab, A in tsqr_inputs(m, n):
        got = lstsq_tsqr_dev(A, B).run(ctx)
        ref = with_option(ctx, "TSQR_HOUSEHOLDER", lstsq_tsqr_dev(A, B).run, ctx)
        for key in got:
            same_bits(f"lstsq_tsqr {label} {lab} {key}", got[key], ref[key])


# ----------------------------------------------------------------------------- 6. GEMM with beta = 0
@pytest.mark.parametrize("label,ta,tb,shape", GEMM_CASES, ids=[c[0] for c in GEMM_CASES])
def test_gemm_beta_zero_does_not_read_c(ctx, label, ta, tb, shape):
    M, N, K = shape
    rng = np.random.default_rng(M + N + K)
    A = rng.standard_normal((K, M) if ta else (M, K))
    B = rng.standard_normal((N, K) if tb else (K, N))
    dA, dB = ctx.upload(A), ctx.upload(B)
    route = gemm_route(ta, tb, M, N, K, 0.0, ctx.props()["sm_count"])
    assert route == label.split("_")[0]
    for alpha in (1.0, -0.75, 0.0):
        res = {}
        for c0 in (0.0, np.nan, np.inf, -np.inf):
            dC = ctx.upload(np.full((M, N), c0))
            _, nl = counted(ctx, ctx.call, "lq_gemm_dev", ta, tb, M, N, K, alpha, dA.ptr, A.shape[1], dB.ptr, B.shape[1], 0.0,
                            dC.ptr, N)
            assert nl == (2 if route in ("split", "remainder") else 1), (route, nl)
            res[c0] = ctx.download(dC, (M, N))
        assert np.isfinite(res[0.0]).all(), (label, alpha)
        for c0 in (np.nan, np.inf, -np.inf):
            same_bits(f"gemm {label} alpha={alpha} C={c0}", res[c0], res[0.0])

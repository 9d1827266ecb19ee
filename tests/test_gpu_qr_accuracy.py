"""Backward error, orthogonality and the forward error of R of every QR route, in units of u = 2^-53.

``test_gpu_routes.py`` proves which kernel each shape reaches and holds Q and R to the reference at 1e-10; that bar is
about 1e6 u, so a kernel that lost eight bits in a reflector or a normalisation would still pass it.  The bounds here are
those of a correct factorisation, with the size unit s = sqrt(m n) u, and every error is evaluated in extended precision
(``_hp``: 80-bit long double, or mpmath where long double is plain double):

1. columnwise backward error  max_j ||a_j - Q r_j|| / ||a_j||   <= C_BWD s   (not for MGS with reorth=True, which returns
   the second sweep's R, linalg/qr.py:46-47);
2. orthogonality  max |Q^T Q - I| <= C_ORTH s (Householder, TSQR, MGS with reorth).  Single-sweep MGS loses orthogonality
   in proportion to the conditioning (Bjorck), so there the diagonal |q_j^T q_j - 1| <= C_NRM s, which does not depend on
   kappa, and the off-diagonal <= C_MGS s kappa_D;
3. the forward error of R  max_j ||r_j - r^_j|| / ||a_j|| <= C_R s kappa_D, kappa_D = cond(A diag(1 / ||a_j||)), against
   ``hp_householder`` (the reference's signs for Householder, a positive diagonal for MGS and TSQR) where m n^2 <= 2^26,
   against sign-fixed LAPACK with twice the bound beyond.  MGS is invariant under column scaling, so its off-diagonal
   bound uses kappa_D as well;
4. LAPACK's ``np.linalg.qr`` of the same input, signs fixed the same way, meets every bound of the case, which shows that
   the bound is not tighter than the problem.

Where m n > 2^18 the full error matrices are not formed: 1 and 2 are estimated from PROBES seeded Gaussian vectors X as
||(A - QR) X||_F / ||A X||_F (about ||A - QR||_F / ||A||_F, at most the columnwise maximum) and
||Q^T (Q X) - X||_F / (sqrt(n) ||X||_F) (about the root mean square of Q^T Q - I, at most its largest entry).

Inputs, on every route and shape: Gaussian; kappa = 1e4 and 1e12 (geometric spectrum, scaled to sigma_min = 1e-3, far
from the 1e-12 skip / dependence threshold); column norms spread by 10^U(-6, 6) (not powers of two, which are bitwise
invariant and tested in ``test_gpu_scaling.py``); a near-dependent pair a_j = a_i + 1e-7 g.  Householder routes also get a
zero and an exactly dependent column (metrics 1 and 2 only: R is not unique there).

Constants, one per metric and family, the same on every route of the family: at least twice the largest ratio measured on
a B200 (1000 W) over every case of this file, and no smaller than LAPACK's largest ratio on the same inputs, which sets the
MGS constants (Householder-quality factors of 32 x 32 matrices reach 0.34 s on |q_j^T q_j - 1|):

========  ===========  =====  ===========  ==============
constant  family       value  B200 maximum LAPACK maximum
========  ===========  =====  ===========  ==============
C_BWD     Householder  1.25   0.58         0.33
C_ORTH    Householder  1.75   0.84         0.37
C_R       Householder  0.05   0.012        0.029
C_BWD     MGS          0.5    0.094        0.32
C_NRM     MGS          0.5    0.11         0.34
C_MGS     MGS          0.1    0.039        0.0042
C_ORTH    MGS reorth   0.5    0.11         0.34
C_R       MGS          0.025  0.0063       0.0091
C_BWD     TSQR         0.75   0.37         0.14
C_ORTH    TSQR         0.75   0.32         0.16
C_R       TSQR         0.1    0.043        0.033
========  ===========  =====  ===========  ==============

A scaling by (1 + 2^-46) of beta in any one Householder kernel, of 1 / ||v|| in the 32 x 32 MGS kernel or of the Cholesky
row scale of CholeskyQR2 exceeds these bounds 2-25 times on its route; one Newton step fewer in the 32 x 32 Householder
kernel, about 2000 times.

The Newton-refined reciprocal, rsqrt and sqrt that build ||x||, beta and 1 / ||v|| in these kernels are measured by
``lq_probe`` kinds 10-16 (``probe_seed_accuracy_kernel``).  On a B200: the MUFU rcp and rsqrt seeds 9.9e-7 and 9.2e-7
(about 2^-20); the refined rcp and sqrt exact on every sample, rsqrt 2.56e-16 and the two-step rsqrt 2.68e-16 (2.3 u and
2.4 u against a reference that is itself rounded twice), the two-step rcp exact.
"""
import numpy as np
import pytest

import linalg_b200 as lb
from test_gpu_routes import (U64, _hp, _resolve, assert_route, conditioned, counted, hh_qr_route,
                             hp_householder, mgs_qr_route)
from test_gpu_tallskinny_routes import assert_within, tsqr_route, with_option

pytestmark = pytest.mark.gpu

C_BWD = {"hh": 1.25, "mgs": 0.5, "tsqr": 0.75}
C_ORTH = {"hh": 1.75, "mgs": 0.5, "tsqr": 0.75}      # MGS: with reorth only
C_R = {"hh": 0.05, "mgs": 0.025, "tsqr": 0.1}
C_NRM = 0.5         # single-sweep MGS, |q_j^T q_j - 1|
C_MGS = 0.1         # single-sweep MGS, off-diagonal of Q^T Q, per unit of kappa_D

FULL_MN = 1 << 18       # beyond: metrics 1 and 2 from probe vectors
HP_R_MNN = 1 << 26      # beyond: R against LAPACK, with twice the bound
PROBES = 4

KINDS = ["gaussian", "kappa1e4", "kappa1e12", "mixed_norms", "near_dependent"]
HH_KINDS = KINDS + ["zero_col", "dependent_col"]
NOT_UNIQUE = {"zero_col", "dependent_col"}


def make_input(kind, m, n, rng):
    """One input of the kind, or None where the kind needs two columns and n == 1."""
    if kind.startswith("kappa"):
        kappa = float(kind[5:])
        return 1e-3 * kappa * conditioned(rng, m, n, kappa)
    A = rng.standard_normal((m, n))
    if kind == "mixed_norms":
        return A * 10.0 ** rng.uniform(-6.0, 6.0, n)
    if kind == "gaussian":
        return A
    if n < 2:
        return None
    i, j = n // 3, (2 * n) // 3 if n > 2 else 1
    if kind == "near_dependent":
        A[:, j] = A[:, i] + 1e-7 * rng.standard_normal(m)
    elif kind == "zero_col":
        A[:, j] = 0.0
    elif kind == "dependent_col":
        A[:, j] = 2.0 * A[:, i]
    else:
        raise KeyError(kind)
    return A


def inputs(kinds, m, n, seed):
    rng = np.random.default_rng(seed)
    out = [(k, make_input(k, m, n, rng)) for k in kinds]
    return [(k, A) for k, A in out if A is not None]


def _ratio_max(num, den):
    """max num / den, with 0 / 0 = 0."""
    return float(np.max(np.divide(num, den, out=np.where(num > 0, np.inf, 0.0), where=den > 0)))


def _hp_colnorm2(E):
    return np.sum(E * E, axis=0).astype(np.float64)


def factor_errors(A, Q, R, family, *, reorth=False, Rref=None, kappa_d=None, ref_factor=1):
    """(error, bound) of every metric that applies; Rref (signs fixed to the family's convention) adds the R check."""
    m, n = A.shape
    s = np.sqrt(m * n) * U64
    Ah, Qh, Rh = _hp(A), _hp(Q), _hp(R)
    out = {}
    mgs_single = family == "mgs" and not reorth
    if m * n <= FULL_MN:
        if not (family == "mgs" and reorth):
            err = np.sqrt(_hp_colnorm2(Ah - Qh @ Rh))
            out["bwd"] = (_ratio_max(err, np.linalg.norm(A, axis=0)), C_BWD[family] * s)
        G = np.abs((Qh.T @ Qh - _hp(np.eye(n))).astype(np.float64))
        if mgs_single:
            out["nrm"] = (np.max(np.diag(G)), C_NRM * s)
            if n > 1 and kappa_d is not None:
                out["offdiag"] = (np.max(G - np.diag(np.diag(G))), C_MGS * s * kappa_d)
        else:
            out["orth"] = (np.max(G), C_ORTH[family] * s)
    else:
        assert not mgs_single, "single-sweep MGS is checked entrywise"
        X = np.random.default_rng(m + 7 * n).standard_normal((n, PROBES))
        Xh = _hp(X)
        AX = Ah @ Xh
        E = AX - Qh @ (Rh @ Xh)
        out["bwd_est"] = (np.sqrt(float(np.sum(E * E)) / float(np.sum(AX * AX))), C_BWD[family] * s)
        Y = Qh.T @ (Qh @ Xh) - Xh
        out["orth_est"] = (np.sqrt(float(np.sum(Y * Y)) / (n * float(np.sum(X * X)))), C_ORTH[family] * s)
    if Rref is not None and not (family == "mgs" and reorth):
        err = np.linalg.norm(R - Rref, axis=0)
        out["R"] = (_ratio_max(err, np.linalg.norm(A, axis=0)), ref_factor * C_R[family] * s * kappa_d)
    return out


def sign_flips(R, signs):
    """+-1 per row of R such that the flipped diagonal has the given signs where both are non-zero."""
    return np.where(np.sign(np.diag(R)) * signs < 0, -1.0, 1.0)


def check_qr(label, A, Q, R, family, kind, reorth=False):
    """Every metric of the case on the route's Q, R and on LAPACK's factors of the same A."""
    m, n = A.shape
    assert np.all(np.isfinite(Q)) and np.all(np.isfinite(R)), label
    assert np.all(np.tril(R, -1) == 0.0), label
    Rref = kappa_d = None
    ref_factor = 1
    # the reference's signs for Householder (the route's own where R is not unique or not computed here), else diag > 0
    signs = np.sign(np.diag(R)) if family == "hh" else np.ones(n)
    if kind not in NOT_UNIQUE:
        sv = np.linalg.svd(A / np.linalg.norm(A, axis=0), compute_uv=False)
        kappa_d = sv[0] / sv[-1]
        if m * n * n <= HP_R_MNN:
            Rref = hp_householder(A)[1]
            if family == "hh":
                signs = np.sign(np.diag(Rref))
        else:
            Rref, ref_factor = np.linalg.qr(A, mode="r"), 2
        Rref = sign_flips(Rref, signs)[:, None] * Rref
    Ql, Rl = np.linalg.qr(A)
    d = sign_flips(Rl, signs)
    Ql, Rl = Ql * d, d[:, None] * Rl
    kw = dict(reorth=reorth, Rref=Rref, kappa_d=kappa_d, ref_factor=ref_factor)
    assert_within(f"lapack {label}", **factor_errors(A, Ql, Rl, family, **kw))
    assert_within(label, **factor_errors(A, Q, R, family, **kw))


# ----------------------------------------------------------------------------- the accuracy probe
def test_seed_and_newton_accuracy_probe(ctx):
    """lq_probe kinds 10-16: the raw MUFU rcp / rsqrt seeds (10, 11) are measured (coarser than 2^-40, so one Newton step
    fewer would leave errors far above u), the Newton-refined rcp, rsqrt, sqrt and the two-step rcp / rsqrt that the QR
    kernels use (12-16) are within 2.5 u relative.  The probe's rsqrt reference 1.0 / sqrt(x) is itself rounded twice (up
    to 1 u), which is why 2 u is not the bound there."""
    v = {k: ctx.probe(k) for k in range(10, 17)}
    assert all(np.isfinite(x) for x in v.values()), v
    assert v[10] > 2.0 ** -40 and v[11] > 2.0 ** -40, v
    assert all(v[k] <= 2.5 * U64 for k in range(12, 17)), v


# ----------------------------------------------------------------------------- batched 32 x 32 kernels
def slot_batches(kinds, per_warp, full_warps, tail):
    """Batches of full_warps warps of per_warp matrices plus a partial warp of `tail`: matrix i of warp w sits in slot
    s = i % per_warp and has kind (w + s + offset) % len(kinds).  Every kind meets every slot within the first
    len(kinds) warps; the offsets step by `tail`, so that every kind also lands in the partial last warp."""
    nk = len(kinds)
    batch = per_warp * full_warps + tail
    assert full_warps >= nk and 0 < tail < per_warp
    for offset in range(0, nk, tail):
        yield offset, [kinds[(i // per_warp + i % per_warp + offset) % nk] for i in range(batch)]


def run_slot_batch(ctx, fn, kinds_of, seed, **kw):
    rng = np.random.default_rng(seed)
    A = np.stack([make_input(k, 32, 32, rng) for k in kinds_of])
    (Q, R), nl = counted(ctx, fn, A, ctx=ctx, **kw)
    return A, Q, R, nl


def test_householder_qr32_every_slot(ctx):
    """hh_qr32_c8_kernel: 4 matrices per warp, 8 warps per CTA, the Q phase pipelined over the warp's four slots.  A batch
    of 2 x 32 + 15 leaves the last CTA and its last warp partial; every input kind runs in each of the four slots and in
    the partial warp."""
    smem = ctx.props()["max_smem"]
    assert hh_qr_route(32, 32, smem, batched=True) == "qr32"
    for offset, kinds_of in slot_batches(HH_KINDS, 4, 2 * 8 + 3, 3):
        A, Q, R, nl = run_slot_batch(ctx, lb.householder_qr_batched, kinds_of, 3200 + offset)
        assert len(A) == 2 * 32 + 15
        assert_route("qr32", nl, len(A))
        for i, kind in enumerate(kinds_of):
            check_qr(f"qr32 hh #{i} slot {i % 4} {kind}", A[i], Q[i], R[i], "hh", kind)


@pytest.mark.parametrize("reorth", [False, True])
def test_mgs_qr32_every_slot(ctx, reorth):
    """mgs_qr32_kernel: 2 matrices per warp, 2 warps per block (api_batched.cu).  A batch of 2 x 4 + 3 leaves the last block
    and its last warp partial; every input kind runs in both slots and in the partial warp."""
    smem = ctx.props()["max_smem"]
    assert mgs_qr_route(32, 32, smem) == "qr32"
    for offset, kinds_of in slot_batches(KINDS, 2, 2 * 2 + 1, 1):
        A, Q, R, nl = run_slot_batch(ctx, lb.qr_batched, kinds_of, 3300 + offset, reorth=reorth)
        assert len(A) == 2 * 4 + 3
        assert_route("qr32", nl, len(A))
        for i, kind in enumerate(kinds_of):
            check_qr(f"qr32 mgs #{i} slot {i % 2} reorth={reorth} {kind}", A[i], Q[i], R[i], "mgs", kind, reorth)


# ----------------------------------------------------------------------------- Householder: one CTA and blocked
def _id(shape):
    return shape.replace(":", "_") if isinstance(shape, str) else "x".join(map(str, shape))


HH_BATCHED = [(33, 32), (65, 64), (100, 80), "hh_square:0", "hh_tall2:0", "hh_square:1", "hh_tall2:1"]
HH_SINGLE = [(64, 64), (4096, 1), (130, 129), (300, 300), (700, 130), (5000, 200), (2100, 2017)]


@pytest.mark.parametrize("shape", HH_BATCHED, ids=_id)
def test_householder_qr_batched_routes(ctx, shape):
    """householder_qr_batched on the one-CTA small_hh_kernel (last fitting shapes included) and, one past the one-CTA
    limit, on the blocked path matrix by matrix: every input kind in one batch."""
    smem = ctx.props()["max_smem"]
    m, n = _resolve(shape, smem)
    route = hh_qr_route(m, n, smem, batched=True)
    assert route == ("blocked" if shape in ("hh_square:1", "hh_tall2:1") else "small"), (shape, route)
    cases = inputs(HH_KINDS, m, n, 41 * m + n)
    A = np.stack([a for _, a in cases])
    (Q, R), nl = counted(ctx, lb.householder_qr_batched, A, ctx=ctx)
    assert_route(route, nl, len(A))
    for i, (kind, Ai) in enumerate(cases):
        check_qr(f"{route} {m}x{n} {kind}", Ai, Q[i], R[i], "hh", kind)


@pytest.mark.parametrize("shape", HH_SINGLE, ids=_id)
def test_householder_qr_single_routes(ctx, shape):
    """householder_qr: the one-CTA kernel for m n <= 4096, beyond it the blocked path: m < 256, padded columns, panels
    taller than 4096 rows (the cluster panel kernel) and Q in two column ranges (2100 x 2017).  6400 x 6400, the two-range
    trailing update, is not run: building its inputs and LAPACK's reference takes the host well over a minute."""
    smem = ctx.props()["max_smem"]
    m, n = shape
    route = hh_qr_route(m, n, smem, batched=False)
    for kind, A in inputs(HH_KINDS, m, n, 43 * m + n):
        (Q, R), nl = counted(ctx, lb.householder_qr, A, ctx=ctx)
        assert_route(route, nl, 1)
        check_qr(f"{route} {m}x{n} {kind}", A, Q, R, "hh", kind)


# ----------------------------------------------------------------------------- MGS: one CTA and large
MGS_SHAPES = ["mgs_square:0", "mgs_tall2:0", "mgs_square:1", "mgs_tall2:1", (700, 300)]


@pytest.mark.parametrize("reorth", [False, True])
@pytest.mark.parametrize("shape", MGS_SHAPES, ids=_id)
def test_mgs_qr_routes(ctx, shape, reorth):
    """qr_batched on small_mgs_kernel (the last fitting shapes) and on the column-by-column large route beyond it."""
    smem = ctx.props()["max_smem"]
    m, n = _resolve(shape, smem)
    route = mgs_qr_route(m, n, smem)
    assert route == ("small" if str(shape).endswith(":0") else "large"), (shape, route)
    cases = inputs(KINDS, m, n, 47 * m + n + reorth)
    A = np.stack([a for _, a in cases])
    (Q, R), nl = counted(ctx, lb.qr_batched, A, reorth=reorth, ctx=ctx)
    assert_route(route, nl, len(A))
    for i, (kind, Ai) in enumerate(cases):
        check_qr(f"{route} {m}x{n} reorth={reorth} {kind}", Ai, Q[i], R[i], "mgs", kind, reorth)


# ----------------------------------------------------------------------------- TSQR
# (4n, n) for n = 17 and 128, a 1-column last BCGS2 panel, BCGS2 with two full panels and with a wider matrix
TSQR_SHAPES = [(68, 17), (2005, 33), (1024, 128), (1000, 129), (600, 300), (2000, 256)]
TSQR_PANEL = 128
TSQR_COND2_MAX = 1e10


def cholqr_cond2(A):
    """The status word of the first Cholesky of every CholeskyQR2 panel (chol_upper128_kernel: max_j G_jj / min_j R_jj^2
    over the panel's columns after the BCGS2 projections), from LAPACK's R: G_jj = ||R[c0:, j]||^2 for panel c0."""
    R = np.linalg.qr(A, mode="r")
    n = R.shape[1]
    worst = 0.0
    for c0 in range(0, n, TSQR_PANEL):
        cols = range(c0, min(n, c0 + TSQR_PANEL))
        g = max(np.sum(R[c0:j + 1, j] ** 2) for j in cols)
        worst = max(worst, g / min(R[j, j] ** 2 for j in cols))
    return worst


@pytest.mark.parametrize("m,n", TSQR_SHAPES)
def test_tsqr_routes(ctx, m, n):
    """lb.tsqr on CholeskyQR2 (n <= 128), BCGS2 (n > 128) and the Householder fallback, which every input whose Cholesky
    pivot ratio reaches 1e10 takes (kappa = 1e12 always): the fallback is bitwise the result under the TSQR_HOUSEHOLDER
    option, the other routes are not."""
    for kind, A in inputs(KINDS, m, n, 53 * m + n):
        cond2 = cholqr_cond2(A)
        # LAPACK's R gives the kernel's status word to far better than this margin (2000 x 256 at kappa 1e12: 1.8e10)
        assert not 1 / 1.5 < cond2 / TSQR_COND2_MAX < 1.5, (m, n, kind, cond2, "too close to the fallback threshold")
        assert kind != "kappa1e12" or cond2 > TSQR_COND2_MAX
        route = "householder" if cond2 > TSQR_COND2_MAX else tsqr_route(m, n)
        Q, R = lb.tsqr(A, ctx=ctx)
        Qh, Rh = with_option(ctx, "TSQR_HOUSEHOLDER", lb.tsqr, A)
        same = np.array_equal(Q, Qh) and np.array_equal(R, Rh)
        assert same == (route == "householder"), (m, n, kind, route)
        assert np.all(np.diag(R) > 0)
        check_qr(f"tsqr {route} {m}x{n} {kind}", A, Q, R, "tsqr", kind)

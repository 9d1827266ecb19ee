"""The rows SURVEY.md section 8(f) marks "next": callers of the hot path, running on the same device kernels.

``project_onto_colspace`` is the reference's ``linalg/projections.py:15-48`` with the switch its own TODO asks for
(``Q, _ = householder_qr(A); return Q @ (Q.T @ b)``, projections.py:23-25); ``pca`` is ``linalg/svd.py:85-123`` on
the A^T A eigen-route of this package instead of LAPACK's SVD.  All matrix products, factorizations and the
eigen-solve run on the GPU through the C ABI; the host only centres the data and assembles the result tuple.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _native as nat
from .qr import householder_qr, householder_qr_batched, qr, qr_batched
from .svd import svd
from .utils import EPS, as_f64_batch, as_f64_matrix


def _matmul(ctx, A: np.ndarray, B: np.ndarray, trans_a: bool = False) -> np.ndarray:
    """op(A) @ B on the device (lq_gemm_dev, FP64 tensor-core GEMM)."""
    A = np.ascontiguousarray(A, dtype=np.float64)
    B = np.ascontiguousarray(B, dtype=np.float64)
    m = A.shape[1] if trans_a else A.shape[0]
    k = A.shape[0] if trans_a else A.shape[1]
    n = B.shape[1]
    if B.shape[0] != k:
        raise ValueError(f"shapes {A.shape} (trans={trans_a}) and {B.shape} not aligned")
    out = np.empty((m, n))
    if m == 0 or n == 0:
        return out
    if k == 0:
        out[:] = 0.0
        return out
    dA, dB, dC = ctx.upload(A), ctx.upload(B), ctx.alloc(out.nbytes)
    ctx.call("lq_gemm_dev", int(trans_a), 0, m, n, k, C.c_double(1.0), dA.ptr, A.shape[1], dB.ptr, n, C.c_double(0.0), dC.ptr, n)
    ctx.download(dC, out.shape, out=out)
    for b in (dA, dB, dC):
        b.free()
    return out


def project_onto_colspace(A, b, *, ctx=None) -> np.ndarray:
    """Orthogonal projection of ``b`` onto the column space of ``A``; shape (m, k) for b of shape (m, k) or (m,)."""
    ctx = ctx if ctx is not None else nat.default_context()
    A = np.asarray(A, dtype=float)
    b = np.asarray(b, dtype=float)
    if b.ndim == 1:
        b = b[:, None]  # projections.py:31-32
    m, n = A.shape
    # scale every column by a power of two to a largest entry in [0.5, 1): exact, the column space is the same, and the
    # QR's absolute 1e-12 skip and the relative rank checks below then see a matrix of unit scale (the projection, like
    # the reference's normal equations, does not depend on the scale of A)
    if A.size:
        A = np.ldexp(A, -np.frexp(np.max(np.abs(A), axis=0))[1])
    if m >= n:
        Q, R = householder_qr(A, ctx=ctx)
        d = np.abs(np.diag(R))
        if n == 0 or d.min() > 1e-12 * max(d.max(), 1e-300):
            return _matmul(ctx, Q, _matmul(ctx, Q, b, trans_a=True))  # Q (Q^T b)
    # dependent columns (the reference falls back to the pseudo-inverse, projections.py:35-37):
    # project onto the left singular vectors that carry the range
    U, s, _ = svd(A, ctx=ctx)
    r = int(np.sum(s > 1e-12 * max(s.max() if s.size else 0.0, 1e-300)))
    Ur = np.ascontiguousarray(U[:, :r])
    return _matmul(ctx, Ur, _matmul(ctx, Ur, b, trans_a=True))


def pca(A, k: int, *, ctx=None):
    """PCA with samples in rows (linalg/svd.py:85-123): returns
    ``(pcs, scores, explained_variance, explained_variance_ratio, total_variance, mean_)``."""
    ctx = ctx if ctx is not None else nat.default_context()
    A = np.asarray(A, dtype=float)
    mean_ = A.mean(axis=0, keepdims=True)
    X = A - mean_
    _, S, Vt = svd(X, ctx=ctx)
    pcs = np.ascontiguousarray(Vt[:k].T)
    scores = _matmul(ctx, X, pcs)
    n_samples = A.shape[0]
    explained_variance = (S[:k] ** 2) / (n_samples - 1)
    total_variance = float(np.sum(S ** 2)) / (n_samples - 1)  # = ||X||_F^2 / (n - 1)
    explained_variance_ratio = explained_variance / total_variance
    return pcs, scores, explained_variance, explained_variance_ratio, total_variance, mean_.ravel()


# ----------------------------------------------------------------------------- 8(f)-4: callers of `qr`
def det_batched(A, *, ctx=None, devices=None) -> np.ndarray:
    """Determinants of a (batch, n, n) array from the batched Householder factorisation:
    ``det(A) = det(Q) det(R) = (-1)^k prod(diag R)``, k = number of reflectors actually applied (a column with
    ``||x|| < 1e-12`` is skipped, linalg/qr.py:79-80, and leaves ``|R[j, j]| < 1e-12``).  A skipped column means the
    matrix is singular at the reference's own absolute threshold (``qr`` would raise "linearly dependent" on it,
    linalg/qr.py:40-41): the determinant is then reported as exactly 0, which sends ``adj`` down the cofactor branch
    like the reference's exact-zero pivots do.  The reference's ``det`` (elimination, out of scope) is only needed by
    ``adj``; this keeps ``adj`` entirely on the hot path's kernels."""
    A = as_f64_batch(A)
    b, m, n = A.shape
    if m != n:
        raise ValueError("A must be a square matrix")
    if n == 0:
        return np.ones(b)
    _, R = householder_qr_batched(A, ctx=ctx, devices=devices)
    d = np.diagonal(R, axis1=1, axis2=2)
    applied = np.sum(np.abs(d) >= EPS, axis=1)
    return np.where(applied == n, np.where(n % 2 == 0, 1.0, -1.0) * np.prod(d, axis=1), 0.0)


def det(A, *, ctx=None) -> float:
    A = as_f64_matrix(A)
    return float(det_batched(A[None], ctx=ctx)[0])


def adj_batched(A, *, ctx=None, devices=None) -> np.ndarray:
    """Adjugate of every ``A[b]`` (linalg/matrix_functions.py:36-63): ``det(A) A^-1`` with ``A^-1 = R^-1 Q^T`` from the
    MGS ``qr`` for the non-singular matrices, cofactor expansion (determinants of the (n-1) x (n-1) minors, one batched
    call) for the matrices whose determinant is exactly 0 -- the reference's branch condition ``d == 0`` (:48)."""
    A = as_f64_batch(A)
    b, m, n = A.shape
    if m != n:
        raise ValueError("A must be a square matrix")
    out = np.empty_like(A)
    if b == 0 or n == 0:
        return out
    d = det_batched(A, ctx=ctx, devices=devices)
    sing = d == 0.0
    idx = np.flatnonzero(~sing)
    if idx.size:
        Q, R = qr_batched(A[idx], ctx=ctx, devices=devices)          # matrix_functions.py:61
        ain = np.linalg.solve(R, np.swapaxes(Q, 1, 2))                # :62 (n x n triangular systems, host LAPACK like upstream)
        out[idx] = d[idx, None, None] * ain
    for i in np.flatnonzero(sing):                                    # :49-58
        if n == 1:
            out[i] = 1.0
            continue
        keep = [np.arange(n) != r for r in range(n)]
        minors = np.stack([A[i][keep[r]][:, keep[c]] for r in range(n) for c in range(n)])
        cof = det_batched(minors, ctx=ctx, devices=devices).reshape(n, n)
        sign = (-1.0) ** np.add.outer(np.arange(n), np.arange(n))
        out[i] = (sign * cof).T
    return out


def adj(A, *, ctx=None) -> np.ndarray:
    """Adjugate (classical adjoint) of a square matrix, ``linalg/matrix_functions.py:36-63`` on the device path."""
    A = np.asarray(A)
    if A.ndim != 2:
        raise ValueError("A must be a square matrix")
    return adj_batched(A.astype(float)[None], ctx=ctx)[0]


def random_nonsingular_qr_batched(n: int, seeds, *, ctx=None, devices=None) -> np.ndarray:
    """``random_nonsingular_qr(n, seed)`` (linalg/qr.py:137-154) for every seed of ``seeds`` in one batched MGS call:
    matrix i is bitwise what the one-matrix drop-in returns for ``seeds[i]`` and equals the reference's
    ``random_nonsingular_qr(n, seeds[i])`` to rounding (same ``default_rng`` draws: A first, then the column scales)."""
    seeds = list(seeds)
    A = np.empty((len(seeds), n, n))
    scales = np.empty((len(seeds), n))
    for i, sd in enumerate(seeds):
        rng = np.random.default_rng(sd)
        A[i] = rng.standard_normal((n, n))
        scales[i] = rng.uniform(0.5, 10.0, size=n)
    if len(seeds) == 0 or n == 0:
        return A
    Q, _ = qr_batched(A, ctx=ctx, devices=devices)
    return Q * scales[:, None, :]

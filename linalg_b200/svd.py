"""Drop-in replacement for ``linalg/svd.py::svd`` -- economy SVD through the A^T A eigen-route.

Gram matrix, Jacobi eigen-solver, descending sort, ``s = sqrt(max(lambda, 0))``, ``U = A V / s``
all run on the device (linalg/svd.py:42-64).  Eigenvector signs are whatever the eigen-solver
produces (the reference inherits LAPACK's), so U and V agree with the reference up to a per-column
sign, which is also how the reference's own test compares them (tests/test_svd.py:31-35).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _native as nat
from .qr import _check_out, _run_batched
from .utils import as_f64_batch


def _complete(ctx, U, m, n, r, seed):
    """linalg/svd.py:67-76: complete U (m, n; its first r columns valid) with an orthonormal basis of the complement, in
    place.  ``seed=None`` draws the m x (n - r) candidate directions on the host exactly like upstream (global np.random);
    an integer generates them on the device.  The projection and both orthonormalisations run on the device."""
    if seed is None:
        Z = np.ascontiguousarray(np.random.randn(m, n - r))
        ctx.call("lq_svd_complete", U.ctypes.data, m, n, r, Z.ctypes.data)
    else:
        ctx.call("lq_svd_complete_seeded", U.ctypes.data, m, n, r, int(seed) & 0xFFFFFFFFFFFFFFFF)


def svd(A, tol: float = 1e-12, *, ctx=None, seed=None):
    """Returns ``(U, s, Vt)``: U (m, n) orthonormal columns, s (n,) descending, Vt (n, n), for m >= n;
    a wide matrix is handled by transposing and swapping roles (linalg/svd.py:37-39).

    ``seed`` only matters for rank-deficient input (linalg/svd.py:67-76): ``None`` (default) draws the candidate
    directions of the orthonormal completion from the global ``np.random`` exactly like upstream (not reproducible);
    an integer generates them on the device (Philox4x32-10), deterministically and without the m x (n - rank) upload."""
    A = np.asarray(A, dtype=float)
    if A.ndim != 2:
        raise ValueError(f"A must be 2-D (got shape {A.shape}); not enough/too many values to unpack")
    m, n = A.shape
    if m < n:
        Vt, s, Ut = svd(A.T, tol, ctx=ctx, seed=seed)
        return Ut.T, s, Vt.T
    A = np.ascontiguousarray(A, dtype=np.float64)
    ctx = ctx if ctx is not None else nat.default_context()
    U = np.empty((m, n))
    s = np.empty(n)
    Vt = np.empty((n, n))
    if n == 0:
        return U, s, Vt
    rank = C.c_int(0)
    ctx.call("lq_svd_gram", A.ctypes.data, m, n, float(tol), U.ctypes.data, s.ctypes.data, Vt.ctypes.data, C.byref(rank))
    r = int(rank.value)
    if r < n:
        _complete(ctx, U, m, n, r, seed)
    return U, s, Vt


def svd_batched(A, tol: float = 1e-12, *, seed=None, out=None, ctx=None, devices=None):
    """``svd`` applied independently to every ``A[i]`` of a (batch, m, n) array: returns U (batch, m, k), s (batch, k)
    descending, Vt (batch, k, n) with k = min(m, n).  Matrix i of the result is ``svd(A[i], tol, seed=seed)``: the rank
    #(s > tol) is decided per matrix, and each rank-deficient matrix gets U's orthonormal completion.  With ``seed=None``
    the candidates are drawn from the global ``np.random`` for the rank-deficient matrices in increasing i, leaving it in
    the state a loop over ``svd`` leaves.

    n <= 32 and m <= 4096 (after transposing a wide batch) run one warp per matrix; other shapes run the single-matrix
    pipeline matrix by matrix, bit for bit ``svd(A[i])``.  The route depends on the shape alone, so a matrix's result does
    not depend on the batch it is in.  ``out=(U, s, Vt)`` receives the result; ``devices=[0, 1, ...]`` splits the batch
    contiguously over several GPUs of this process (bitwise the one-GPU result)."""
    A = as_f64_batch(A)
    b, m, n = A.shape
    k = min(m, n)
    if out is not None:
        U, s, Vt = out
        _check_out(U, (b, m, k))
        _check_out(s, (b, k))
        _check_out(Vt, (b, k, n))
    if m < n:
        Vt_, s_, Ut = svd_batched(np.ascontiguousarray(A.transpose(0, 2, 1)), tol, seed=seed, ctx=ctx, devices=devices)
        U_, Vt_ = Ut.transpose(0, 2, 1), Vt_.transpose(0, 2, 1)
        if out is None:
            return U_, s_, Vt_
        U[...], s[...], Vt[...] = U_, s_, Vt_
        return U, s, Vt
    if out is None:
        U, s, Vt = np.empty((b, m, n)), np.empty((b, n)), np.empty((b, n, n))
    if b == 0 or n == 0:
        return U, s, Vt
    rank = np.zeros(b, dtype=np.int32)
    _run_batched(ctx, devices, b, lambda c, lo, hi: c.call("lq_svd_gram_batched", A[lo:hi].ctypes.data, hi - lo, m, n, float(tol),
                                                           U[lo:hi].ctypes.data, s[lo:hi].ctypes.data, Vt[lo:hi].ctypes.data,
                                                           rank[lo:hi].ctypes.data))
    deficient = np.flatnonzero(rank < n)
    if deficient.size:
        # linalg/svd.py:67-76 for each rank-deficient matrix, in increasing i (the global np.random draws of a loop over svd)
        cctx = ctx if ctx is not None else (nat.default_context() if devices is None else nat.device_context(devices[0]))
        for i in deficient:
            _complete(cctx, U[i], m, n, int(rank[i]), seed)
    return U, s, Vt

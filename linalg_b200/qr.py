"""Drop-in replacements for ``linalg/qr.py`` running on a B200 through the C ABI.

Same names, argument meaning, shapes, sign conventions and error behaviour as the reference
(``qr`` = modified Gram-Schmidt, linalg/qr.py:14-49; ``householder_qr`` :52-100;
``least_squares_qr`` :103-119; ``least_squares_householder_qr`` :122-134), NumPy arrays in and
out.  There is no CPU implementation here: without the CUDA library and a B200 every call raises.
"""
from __future__ import annotations

import ctypes as C
from typing import Tuple

import numpy as np

from . import _native as nat
from .utils import as_f64_batch, as_f64_matrix

_DEPENDENT = "Input vectors are linearly dependent"  # linalg/qr.py:41


def _ctx(ctx):
    return ctx if ctx is not None else nat.default_context()


def _ptr(a: np.ndarray):
    return a.ctypes.data


def _run_batched(ctx, devices, batch, fn):
    """``fn(ctx, lo, hi)`` on the whole batch with one context, or on contiguous slices of it with one context and one
    host thread per device of ``devices`` (optional kwarg of the ``*_batched`` entry points, SURVEY.md section 5)."""
    if devices is None:
        fn(_ctx(ctx), 0, batch)
    else:
        if ctx is not None:
            raise ValueError("pass either ctx= or devices=, not both")
        nat.fan_out(devices, batch, fn)


# ----------------------------------------------------------------------------- a1
def householder_qr(A, *, ctx=None) -> Tuple[np.ndarray, np.ndarray]:
    """Householder QR of an (m, n) matrix, m >= n.  Returns Q (m, n), R (n, n).

    ``R[j, j] = -copysign(||x||, x[0])`` for every column (also the last one of a square
    matrix), columns with ``||x|| < 1e-12`` are skipped, R's strict lower triangle is exactly 0.
    m < n raises ``ValueError`` (the reference dies in a matmul shape check, SURVEY.md 8a).
    """
    A = as_f64_matrix(A)
    m, n = A.shape
    if m < n:
        raise ValueError(f"householder_qr needs m >= n, got {m} x {n} (matmul shape mismatch upstream)")
    Q = np.empty((m, n))
    R = np.empty((n, n))
    if m == 0 or n == 0:
        return Q, R
    _ctx(ctx).call("lq_householder_qr", _ptr(A), m, n, _ptr(Q), _ptr(R))
    return Q, R


def householder_qr_batched(A, *, out=None, ctx=None, devices=None) -> Tuple[np.ndarray, np.ndarray]:
    """``householder_qr`` applied independently to every ``A[b]`` of a (batch, m, n) array.

    ``devices=[0, 1, ...]`` splits the batch index contiguously over several GPUs of this process (no communication);
    the result is bitwise the one-GPU result."""
    A = as_f64_batch(A)
    b, m, n = A.shape
    if m < n:
        raise ValueError(f"householder_qr needs m >= n, got {m} x {n}")
    if out is None:
        Q, R = np.empty((b, m, n)), np.empty((b, n, n))
    else:
        Q, R = out
        _check_out(Q, (b, m, n))
        _check_out(R, (b, n, n))
    if b and m and n:
        _run_batched(ctx, devices, b, lambda c, lo, hi: c.call("lq_householder_qr_batched", _ptr(A[lo:hi]), hi - lo, m, n,
                                                               _ptr(Q[lo:hi]), _ptr(R[lo:hi])))
    return Q, R


# ----------------------------------------------------------------------------- a2
def qr(A, reorth: bool = False, *, ctx=None) -> Tuple[np.ndarray, np.ndarray]:
    """Modified Gram-Schmidt QR (``diag(R) > 0``).

    ``reorth=True`` runs the second sweep over Q and returns the SECOND sweep's R, exactly like
    the reference (its closure overwrites R, linalg/qr.py:46-47).  A column whose remaining norm
    is below 1e-12 raises ``ValueError("Input vectors are linearly dependent")``.
    """
    A = as_f64_matrix(A)
    m, n = A.shape
    Q = np.empty((m, n))
    R = np.empty((n, n))
    if n == 0:
        return Q, R
    if m == 0:
        raise ValueError(_DEPENDENT)
    info = np.zeros(1, dtype=np.int32)
    _ctx(ctx).call("lq_mgs_qr", _ptr(A), m, n, int(bool(reorth)), _ptr(Q), _ptr(R), _ptr(info))
    if info[0] != 0:
        raise ValueError(_DEPENDENT)
    return Q, R


def qr_batched(A, reorth: bool = False, *, out=None, ctx=None, devices=None) -> Tuple[np.ndarray, np.ndarray]:
    A = as_f64_batch(A)
    b, m, n = A.shape
    if out is None:
        Q, R = np.empty((b, m, n)), np.empty((b, n, n))
    else:
        Q, R = out
        _check_out(Q, (b, m, n))
        _check_out(R, (b, n, n))
    info = np.zeros(max(b, 1), dtype=np.int32)
    if b and m and n:
        _run_batched(ctx, devices, b, lambda c, lo, hi: c.call("lq_mgs_qr_batched", _ptr(A[lo:hi]), hi - lo, m, n, int(bool(reorth)),
                                                               _ptr(Q[lo:hi]), _ptr(R[lo:hi]), _ptr(info[lo:hi])))
    if np.any(info[:b] != 0):
        raise ValueError(_DEPENDENT)
    return Q, R


# ----------------------------------------------------------------------------- a3 / a4
def _rhs_2d(b, m):
    b = np.asarray(b)
    if b.ndim == 1:
        if b.shape[0] != m:
            raise ValueError(f"shapes ({m},?) and {b.shape} not aligned")
        return np.ascontiguousarray(b.reshape(m, 1), dtype=np.float64), True
    if b.ndim == 2:
        if b.shape[0] != m:
            raise ValueError(f"shapes ({m},?) and {b.shape} not aligned")
        return np.ascontiguousarray(b, dtype=np.float64), False
    raise ValueError(f"b must be 1-D or 2-D, got shape {b.shape}")


def least_squares_householder_qr(A, b, *, ctx=None) -> np.ndarray:
    """min ||Ax - b||_2 via Householder QR; returns (n,) for a vector b, (n, k) for a matrix."""
    A = as_f64_matrix(A)
    m, n = A.shape
    if m < n:
        raise ValueError(f"least_squares_householder_qr needs m >= n, got {m} x {n}")
    B, was_vec = _rhs_2d(b, m)
    k = B.shape[1]
    X = np.empty((n, k))
    info = np.zeros(1, dtype=np.int32)
    if n and k:
        _ctx(ctx).call("lq_lstsq_householder_batched_info", _ptr(A), _ptr(B), 1, m, n, k, _ptr(X), _ptr(info))
    if info[0] != 0:
        raise np.linalg.LinAlgError("Singular matrix")  # np.linalg.solve(R, y) upstream, linalg/qr.py:134
    return X.reshape(n) if was_vec else X


def least_squares_qr(A, b, *, ctx=None) -> np.ndarray:
    """min ||Ax - b||_2 via MGS QR.  The result is ALWAYS 1-D (``.ravel()``, linalg/qr.py:119):
    for k right-hand sides it has n*k entries in row-major (n, k) order."""
    A = as_f64_matrix(A)
    m, n = A.shape
    B, _ = _rhs_2d(b, m)
    k = B.shape[1]
    X = np.empty((n, k))
    info = np.zeros(1, dtype=np.int32)
    if n and k:
        _ctx(ctx).call("lq_lstsq_mgs_batched", _ptr(A), _ptr(B), 1, m, n, k, _ptr(X), _ptr(info))
    if info[0] != 0:
        raise ValueError(_DEPENDENT)
    return X.ravel()


def least_squares_householder_qr_batched(A, B, *, out=None, ctx=None, devices=None) -> np.ndarray:
    """A (batch, m, n), B (batch, m, k) -> X (batch, n, k)."""
    A = as_f64_batch(A)
    B = as_f64_batch(B, "B")
    bsz, m, n = A.shape
    if B.shape[0] != bsz or B.shape[1] != m:
        raise ValueError(f"A {A.shape} and B {B.shape} not aligned")
    if m < n:
        raise ValueError(f"least squares needs m >= n, got {m} x {n}")
    k = B.shape[2]
    X = np.empty((bsz, n, k)) if out is None else out
    _check_out(X, (bsz, n, k))
    info = np.zeros(max(bsz, 1), dtype=np.int32)
    if bsz and n and k:
        _run_batched(ctx, devices, bsz, lambda c, lo, hi: c.call("lq_lstsq_householder_batched_info", _ptr(A[lo:hi]), _ptr(B[lo:hi]),
                                                                 hi - lo, m, n, k, _ptr(X[lo:hi]), _ptr(info[lo:hi])))
    if np.any(info[:bsz] != 0):
        raise np.linalg.LinAlgError("Singular matrix")  # np.linalg.solve(R, y) upstream, linalg/qr.py:134
    return X


def least_squares_qr_batched(A, B, *, out=None, ctx=None, devices=None) -> np.ndarray:
    """Batched MGS least squares; X has shape (batch, n*k) -- each row is the reference's ravel()."""
    A = as_f64_batch(A)
    B = as_f64_batch(B, "B")
    bsz, m, n = A.shape
    if B.shape[0] != bsz or B.shape[1] != m:
        raise ValueError(f"A {A.shape} and B {B.shape} not aligned")
    k = B.shape[2]
    X = np.empty((bsz, n, k)) if out is None else out
    _check_out(X.reshape(bsz, n, k), (bsz, n, k))
    info = np.zeros(max(bsz, 1), dtype=np.int32)
    if bsz and n and k:
        Xv = X.reshape(bsz, n, k)
        _run_batched(ctx, devices, bsz, lambda c, lo, hi: c.call("lq_lstsq_mgs_batched", _ptr(A[lo:hi]), _ptr(B[lo:hi]), hi - lo, m, n, k,
                                                                 _ptr(Xv[lo:hi]), _ptr(info[lo:hi])))
    if np.any(info[:bsz] != 0):
        raise ValueError(_DEPENDENT)
    return X.reshape(bsz, n * k)


# ----------------------------------------------------------------------------- a7
def tsqr(A, *, ctx=None) -> Tuple[np.ndarray, np.ndarray]:
    """Thin QR of a tall-skinny (m, n) matrix, m >= n, with ``diag(R) > 0`` (the ``qr`` convention)."""
    A = as_f64_matrix(A)
    m, n = A.shape
    if m < n:
        raise ValueError(f"tsqr needs m >= n, got {m} x {n}")
    Q = np.empty((m, n))
    R = np.empty((n, n))
    if n:
        _ctx(ctx).call("lq_tsqr", _ptr(A), m, n, _ptr(Q), _ptr(R))
    return Q, R


def least_squares_tsqr(A, b, *, ctx=None) -> np.ndarray:
    """min ||Ax - b||_2 for a tall-skinny A on the TSQR pipeline (CholeskyQR2 that never forms Q, Householder least squares
    when A is ill-conditioned, nearly square or wider than 128 columns).  The contract of ``least_squares_householder_qr``:
    (n,) for a vector b, (n, k) for a matrix; m < n raises ``ValueError``; an exactly singular R raises
    ``np.linalg.LinAlgError("Singular matrix")``."""
    A = as_f64_matrix(A)
    m, n = A.shape
    if m < n:
        raise ValueError(f"least_squares_tsqr needs m >= n, got {m} x {n}")
    B, was_vec = _rhs_2d(b, m)
    k = B.shape[1]
    X = np.empty((n, k))
    info = np.zeros(1, dtype=np.int32)
    if n and k:
        _ctx(ctx).call("lq_lstsq_tsqr", _ptr(A), m, n, _ptr(B), k, _ptr(X), _ptr(info))
    if info[0] != 0:
        raise np.linalg.LinAlgError("Singular matrix")
    return X.reshape(n) if was_vec else X


def random_nonsingular_qr(n, seed=None, *, ctx=None) -> np.ndarray:
    """Random orthogonal x random non-zero column scales (reference linalg/qr.py:137-154)."""
    rng = np.random.default_rng(seed)
    A = rng.standard_normal((n, n))
    Q, _ = qr(A, ctx=ctx)
    scales = rng.uniform(0.5, 10.0, size=n)
    return np.asarray(Q * scales)


def _check_out(arr, shape):
    if not isinstance(arr, np.ndarray) or arr.dtype != np.float64 or tuple(arr.shape) != tuple(shape) or not arr.flags.c_contiguous:
        raise ValueError(f"out array must be a C-contiguous float64 ndarray of shape {shape}")

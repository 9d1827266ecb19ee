"""linalg_b200 -- B200-native drop-in for the dense-factorisation hot path of BrantleighBunting/linalg.

Same public names as the reference package for this path (``qr``, ``householder_qr``,
``least_squares_qr``, ``least_squares_householder_qr``, ``svd``, ``random_nonsingular_qr``,
``EPS``; reference ``linalg/__init__.py:65-96``) plus the batched / tall-skinny / sharded surface
BASELINE.json asks for.  NumPy in, NumPy out; the work runs in hand-written sm_100a kernels
reached through ``ctypes`` (``include/linalg_b200.h``).  No PyTorch, no Triton, no CPU fallback.
"""
import logging as _logging

from ._native import Context, default_context, pinned_empty
from .qr import (
    householder_qr,
    householder_qr_batched,
    least_squares_householder_qr,
    least_squares_householder_qr_batched,
    least_squares_qr,
    least_squares_qr_batched,
    least_squares_tsqr,
    qr,
    qr_batched,
    random_nonsingular_qr,
    tsqr,
)
from .svd import svd, svd_batched
from .extras import adj, adj_batched, det, det_batched, pca, project_onto_colspace, random_nonsingular_qr_batched
from .utils import EPS, shard_bounds

__all__ = [
    "qr",
    "householder_qr",
    "least_squares_qr",
    "least_squares_householder_qr",
    "random_nonsingular_qr",
    "svd",
    "svd_batched",
    "EPS",
    "qr_batched",
    "householder_qr_batched",
    "least_squares_qr_batched",
    "least_squares_householder_qr_batched",
    "tsqr",
    "least_squares_tsqr",
    "Context",
    "default_context",
    "pinned_empty",
    "shard_bounds",
    "project_onto_colspace",
    "pca",
    "adj",
    "adj_batched",
    "det",
    "det_batched",
    "random_nonsingular_qr_batched",
]

__version__ = "0.1.0"

_logging.getLogger(__name__).addHandler(_logging.NullHandler())  # reference linalg/__init__.py:110-112

#!/usr/bin/env python3
"""Generate tests/golden/hotpath_golden.npz by running the REAL reference.

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden.py <reference checkout>

The reference (BrantleighBunting/linalg) ships no known-answer vectors for
qr / householder_qr / least_squares_* / svd (SURVEY.md section 8c), so the
fixtures are outputs of the unmodified reference functions on seeded float64
inputs.  Inputs replay the reference's own seeded test cases where it has them
(tests/test_svd.py:13-16, 38-42, 60-70; tests/test_qr.py:29) plus the
BASELINE.json shape classes at fixture-friendly sizes.

To keep the file small, the seeded inputs are not stored: ``golden_inputs()``
regenerates them bit for bit (tests/conftest.py checks them against the SHA-1
stored under ``inputs_sha1``).  Only inputs drawn by the reference's own
generator (``random_nonsingular_upper``) are stored with the outputs.
"""
import hashlib
import os
import sys

import numpy as np

PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "hotpath_golden.npz")

QR_CASES = {
    "sq32": (32, 32, 2),
    "sq5": (5, 5, 11),
    "tall8x5": (8, 5, 13),
    "sq20": (20, 20, 40),
    "tall50x10": (50, 10, 60),
    "tall100x10": (100, 10, 7),
    "tall64x16": (64, 16, 21),
    "sq64": (64, 64, 22),
    "tall96x40": (96, 40, 23),
    "one1x1": (1, 1, 24),
    "col7x1": (7, 1, 25),
}
BATCHED32 = 12  # matrices of the cfg2 shape class (the first 12 of a seed-2 draw of 24)


def golden_inputs():
    """Every seeded input of the fixtures, keyed like the fixture file (``<case>/A``, ``<case>/B``, ``<case>/b``)."""
    inp = {}

    # ---- Householder / MGS QR: the three routines see the same matrices
    for name, (m, n, seed) in QR_CASES.items():
        A = np.random.default_rng(seed).standard_normal((m, n))
        for fam in ("hh", "mgs", "mgs_reorth"):
            inp[f"{fam}/{name}/A"] = A
    # Householder edge cases: a zero column (skip branch, qr.py:79-80), negative
    # pivots, an already upper-triangular matrix, integer dtype input.
    A = np.random.default_rng(31).standard_normal((12, 6))
    A[:, 2] = 0.0
    inp["hh/zero_col/A"] = A
    A = np.random.default_rng(32).standard_normal((9, 9))
    A[3:, 3] = 0.0
    inp["hh/partial_zero/A"] = A
    inp["hh/upper_tri/A"] = np.triu(np.random.default_rng(33).uniform(-5, 5, (10, 10)))
    inp["hh/all_zero/A"] = np.zeros((6, 4))
    inp["hh/integers/A"] = np.random.default_rng(34).integers(-9, 10, (16, 8)).astype(np.float64)
    # batched 32x32 (cfg2 shape class), seed 2 stream
    inp["batched32/A"] = np.random.default_rng(2).standard_normal((24, 32, 32))[:BATCHED32]

    # ---- least squares (ls/upper50_* come from the reference's generator and are stored)
    inp["ls/cfg3/A"] = np.random.default_rng(3).standard_normal((2, 256, 64))
    inp["ls/cfg3/B"] = np.random.default_rng(4).standard_normal((2, 256, 16))
    A = np.random.default_rng(5).standard_normal((40, 12))
    inp["ls/vec40x12/A"] = inp["ls/mat40x12x3/A"] = A
    inp["ls/vec40x12/b"] = np.random.default_rng(6).standard_normal(40)
    inp["ls/mat40x12x3/b"] = np.random.default_rng(7).standard_normal((40, 3))

    # ---- svd
    for m, n in [(8, 5), (20, 20), (50, 10)]:  # tests/test_svd.py:13-16
        inp[f"svd/recon_{m}x{n}/A"] = np.random.default_rng(seed=m + n).normal(size=(m, n))
    for m, n in [(12, 7), (30, 15)]:  # tests/test_svd.py:38-42
        inp[f"svd/np_{m}x{n}/A"] = np.random.default_rng(seed=4 * m + n).standard_normal(size=(m, n))
    for k in (0, 1, 3):  # tests/test_svd.py:60-70 (U's completion columns are random upstream)
        A = np.random.default_rng(123 + k).normal(size=(10, 7))
        if k:
            A[:, -k:] = 0.0
        inp[f"svd/rankdef_{k}/A"] = A
    inp["svd/wide_5x9/A"] = np.random.default_rng(50).standard_normal((5, 9))  # wide -> transpose branch svd.py:37-39
    A = np.random.default_rng(51).standard_normal((1024, 128))  # cfg5 shape class, reduced rows
    inp["svd/tall_1024x128/A"] = A
    inp["tsqr/mgs_1024x64/A"] = A[:1024, :64]
    return {k: np.array(v, dtype=np.float64, order="C") for k, v in inp.items()}  # one private copy per key


def inputs_sha1(inputs):
    """SHA-1 over the names, shapes and bytes of ``inputs`` (as uint8, so it can live in the .npz)."""
    h = hashlib.sha1()
    for k in sorted(inputs):
        v = np.ascontiguousarray(inputs[k], dtype=np.float64)
        h.update(k.encode() + repr(v.shape).encode() + v.tobytes())
    return np.frombuffer(h.digest(), dtype=np.uint8)


def main(ref):
    sys.path.insert(0, ref)
    sys.dont_write_bytecode = True
    from linalg.qr import householder_qr, least_squares_householder_qr, least_squares_qr, qr
    from linalg.svd import svd
    from linalg.utils import random_nonsingular_upper

    inp = golden_inputs()
    out = {}

    def put(name, **arrays):
        for k, v in arrays.items():
            out[f"{name}/{k}"] = np.ascontiguousarray(np.asarray(v, dtype=np.float64))

    for name in QR_CASES:
        A = inp[f"hh/{name}/A"]
        Q, R = householder_qr(A)
        put(f"hh/{name}", Q=Q, R=R)
        Q, R = qr(A)
        put(f"mgs/{name}", Q=Q, R=R)
        Q, R = qr(A, reorth=True)
        put(f"mgs_reorth/{name}", Q=Q, R=R)
    for name in ("zero_col", "partial_zero", "upper_tri", "all_zero", "integers"):
        Q, R = householder_qr(inp[f"hh/{name}/A"])
        put(f"hh/{name}", Q=Q, R=R)
    A = inp["batched32/A"]
    put(
        "batched32",
        Q_hh=np.stack([np.ascontiguousarray(householder_qr(a)[0]) for a in A]),
        R_hh=np.stack([householder_qr(a)[1] for a in A]),
        Q_mgs=np.stack([qr(a)[0] for a in A]),
        R_mgs=np.stack([qr(a)[1] for a in A]),
    )

    for i in range(3):  # tests/test_qr.py:23-47 style, seeded
        U = random_nonsingular_upper(50, seed=100 + i)
        x_true = np.random.default_rng(200 + i).random(50)
        b = U @ x_true
        put(f"ls/upper50_{i}", A=U, b=b, x_hh=least_squares_householder_qr(U, b), x_mgs=least_squares_qr(U, b))
    A, B = inp["ls/cfg3/A"], inp["ls/cfg3/B"]
    put(
        "ls/cfg3",
        X_hh=np.stack([least_squares_householder_qr(A[i], B[i]) for i in range(2)]),
        X_mgs=np.stack([least_squares_qr(A[i], B[i]) for i in range(2)]),
    )
    for name in ("vec40x12", "mat40x12x3"):
        A, b = inp[f"ls/{name}/A"], inp[f"ls/{name}/b"]
        put(f"ls/{name}", x_hh=least_squares_householder_qr(A, b), x_mgs=least_squares_qr(A, b))

    for name in ("recon_8x5", "recon_20x20", "recon_50x10", "np_12x7", "np_30x15",
                 "rankdef_0", "rankdef_1", "rankdef_3", "wide_5x9"):
        np.random.seed(999)  # the rank-deficient completion draws from the global state
        U, s, Vt = svd(inp[f"svd/{name}/A"])
        put(f"svd/{name}", U=U, s=s, Vt=Vt)
    _, s, Vt = svd(inp["svd/tall_1024x128/A"])
    put("svd/tall_1024x128", s=s, Vt=Vt)  # U omitted; checked through invariants
    _, R = qr(inp["tsqr/mgs_1024x64/A"])
    put("tsqr/mgs_1024x64", R=R)

    out["inputs_sha1"] = inputs_sha1(inp)
    np.savez_compressed(PATH, **out)
    print(f"wrote {PATH}: {len(out)} arrays, {os.path.getsize(PATH)/1e6:.2f} MB")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(sys.argv[1])

#!/usr/bin/env python3
"""Batched Householder least squares through the host-pointer entry point, from pinned buffers.

least_squares_householder_qr_batched (lq_lstsq_householder_batched_info) on the cfg3 shape, 256 x 64 with 16 right-hand
sides: by default 2^14 systems (2.7 GB of A and B up, 134 MB of X down, 15 pipeline chunks), with A, B and X in
page-locked NumPy arrays.  Host clock around each call, which returns when X is on the host; min and median of the
repetitions after warm-ups.  The bare copies of the same bytes give the host copy ceiling.  X is checked against the
device entry point bit for bit before anything is printed.  The card's name and power limit are printed with the numbers.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import linalg_b200 as lb  # noqa: E402
from linalg_b200 import _native as nat  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines() if q.returncode == 0 else ["unknown"]


def seconds(fn, warmup, reps):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return ts


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--systems", type=int, default=1 << 14)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the JSON result here")
    a = ap.parse_args()
    b, m, n, k = a.systems, 256, 64, 16
    ctx = lb.default_context()
    rng = np.random.default_rng(3)
    A, B, X = nat.pinned_empty((b, m, n)), nat.pinned_empty((b, m, k)), nat.pinned_empty((b, n, k))
    A[...] = rng.standard_normal((b, m, n))
    B[...] = rng.standard_normal((b, m, k))

    ts = seconds(lambda: lb.least_squares_householder_qr_batched(A, B, out=X, ctx=ctx), a.warmup, a.reps)
    dA, dB, dX, dI = ctx.upload(A), ctx.upload(B), ctx.alloc(X.nbytes), ctx.alloc(4 * b)
    ctx.call("lq_lstsq_householder_batched_info_dev", dA.ptr, dB.ptr, b, m, n, k, dX.ptr, dI.ptr)
    if not np.array_equal(X, ctx.download(dX, X.shape)):
        raise SystemExit("lstsq_host_bench: the host-pointer X differs from the device entry point's")

    def copies():
        ctx.call("lq_memcpy_h2d", dA.ptr, A.ctypes.data, A.nbytes)
        ctx.call("lq_memcpy_h2d", dB.ptr, B.ctypes.data, B.nbytes)
        ctx.call("lq_memcpy_d2h", X.ctypes.data, dX.ptr, X.nbytes)
        ctx.sync()

    tc = seconds(copies, 1, a.reps)
    res = {"card": card(), "shape": [b, m, n, k], "api": "least_squares_householder_qr_batched (pinned host buffers)",
           "host_ptr_ms_min": min(ts) * 1e3, "host_ptr_ms_median": statistics.median(ts) * 1e3,
           "systems_per_s": b / min(ts), "bare_copies_ms_min": min(tc) * 1e3, "copy_bound_share": min(tc) / min(ts)}
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()

#!/usr/bin/env python3
"""First GPU bring-up: probes + batched 32x32 kernels + small kernels vs the oracle.

Run on the GPU box:  python tools/gpu_check1.py > gpurun_out/check1.log 2>&1
"""
import json
import os
import sys
import time
import traceback

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from linalg_b200 import _native as nat  # noqa: E402
from oracle import linalg_oracle as orc  # noqa: E402

out = {}
ctx = nat.Context(0)
print("props", ctx.props(), flush=True)
out["props"] = ctx.props()


def section(name):
    print(f"\n===== {name} =====", flush=True)


def guarded(fn):
    try:
        fn()
    except Exception:
        traceback.print_exc()
        sys.stdout.flush()


# ------------------------------------------------------------------ probes
def probes():
    section("probes")
    for kind, name in [(0, "dfma_tflops"), (1, "dmma_tflops"), (3, "mixed_tflops"), (2, "copy_gbs")]:
        vals = [ctx.probe(kind) for _ in range(3)]
        print(name, vals, flush=True)
        out[name] = max(vals)


guarded(probes)


# ------------------------------------------------------------------ batched 32x32 correctness
def hh32_correct():
    section("hh32 correctness")
    nb = 1000  # not a multiple of the per-block matrix count -> exercises the tail
    A = np.random.default_rng(2).standard_normal((nb, 32, 32))
    A[5, :, 7] = 0.0  # zero column -> skip branch
    A[6] = np.triu(A[6])
    Qo, Ro = orc.householder_qr_batched(A[:64])
    dA = ctx.upload(A)
    dQ = ctx.alloc(A.nbytes)
    dR = ctx.alloc(A.nbytes)
    ctx.call("lq_memset", dQ.ptr, 0xFF, A.nbytes)
    ctx.call("lq_memset", dR.ptr, 0xFF, A.nbytes)
    ctx.call("lq_householder_qr_batched_dev", dA.ptr, nb, 32, 32, dQ.ptr, dR.ptr, 0)
    ctx.sync()
    Q = ctx.download(dQ, A.shape)
    R = ctx.download(dR, A.shape)
    eq = orc.rel_max_err(Q[:64], Qo)
    er = orc.rel_max_err(R[:64], Ro)
    resid = max(orc.qr_residual(A[i], Q[i], R[i]) for i in range(nb))
    orth = orc.orth_error(Q)
    low = float(np.max(np.abs(np.tril(R, -1))))
    out["hh32_correct"] = dict(q=eq, r=er, resid=resid, orth=orth, lower=low)
    print(out["hh32_correct"], flush=True)


guarded(hh32_correct)


def mgs32_correct():
    section("mgs32 correctness")
    nb = 777
    A = np.random.default_rng(3).standard_normal((nb, 32, 32))
    dA = ctx.upload(A)
    dQ = ctx.alloc(A.nbytes)
    dR = ctx.alloc(A.nbytes)
    dI = ctx.alloc(nb * 4)
    for reorth in (0, 1):
        ctx.call("lq_mgs_qr_batched_dev", dA.ptr, nb, 32, 32, reorth, dQ.ptr, dR.ptr, dI.ptr)
        ctx.sync()
        Q = ctx.download(dQ, A.shape)
        R = ctx.download(dR, A.shape)
        info = ctx.download(dI, (nb,), np.int32)
        Qo, Ro = orc.mgs_qr_batched(A[:48], bool(reorth))
        r = dict(q=orc.rel_max_err(Q[:48], Qo), r=orc.rel_max_err(R[:48], Ro), orth=orc.orth_error(Q),
                 info_nonzero=int(np.count_nonzero(info)))
        if not reorth:
            r["resid"] = max(orc.qr_residual(A[i], Q[i], R[i]) for i in range(nb))
        print("reorth", reorth, r, flush=True)
        out[f"mgs32_reorth{reorth}"] = r
    # dependent columns -> info
    A2 = A[:4].copy()
    A2[1, :, 9] = A2[1, :, 3] * 2.0
    dA2 = ctx.upload(A2)
    ctx.call("lq_mgs_qr_batched_dev", dA2.ptr, 4, 32, 32, 0, dQ.ptr, dR.ptr, dI.ptr)
    ctx.sync()
    print("info for dependent col 9 in matrix 1:", ctx.download(dI, (4,), np.int32), flush=True)


guarded(mgs32_correct)


# ------------------------------------------------------------------ small generic kernels
def small_correct():
    section("generic small kernels")
    res = {}
    for (m, n) in [(1, 1), (7, 1), (8, 5), (20, 20), (50, 10), (100, 10), (64, 16), (64, 64), (96, 40), (33, 32),
                   (128, 100)]:
        nb = 5
        A = np.random.default_rng(100 + m + n).standard_normal((nb, m, n))
        dA = ctx.upload(A)
        dQ = ctx.alloc(A.nbytes)
        dR = ctx.alloc(nb * n * n * 8)
        dI = ctx.alloc(nb * 4)
        ctx.call("lq_householder_qr_batched_dev", dA.ptr, nb, m, n, dQ.ptr, dR.ptr, 0)
        ctx.sync()
        Q = ctx.download(dQ, A.shape)
        R = ctx.download(dR, (nb, n, n))
        Qo, Ro = orc.householder_qr_batched(A)
        e1 = dict(q=orc.rel_max_err(Q, Qo), r=orc.rel_max_err(R, Ro))
        ctx.call("lq_mgs_qr_batched_dev", dA.ptr, nb, m, n, 0, dQ.ptr, dR.ptr, dI.ptr)
        ctx.sync()
        Q = ctx.download(dQ, A.shape)
        R = ctx.download(dR, (nb, n, n))
        Qo, Ro = orc.mgs_qr_batched(A)
        e2 = dict(q=orc.rel_max_err(Q, Qo), r=orc.rel_max_err(R, Ro))
        ctx.call("lq_mgs_qr_batched_dev", dA.ptr, nb, m, n, 1, dQ.ptr, dR.ptr, dI.ptr)
        ctx.sync()
        Q = ctx.download(dQ, A.shape)
        R = ctx.download(dR, (nb, n, n))
        Qo, Ro = orc.mgs_qr_batched(A, True)
        e3 = dict(q=orc.rel_max_err(Q, Qo), r=orc.rel_max_err(R, Ro))
        print((m, n), "hh", e1, "mgs", e2, "mgs_reorth", e3, flush=True)
        res[f"{m}x{n}"] = dict(hh=e1, mgs=e2, mgs_reorth=e3)
    # least squares
    for (m, n, k) in [(50, 50, 1), (40, 12, 3), (256, 64, 16), (100, 30, 7)]:
        nb = 4
        A = np.random.default_rng(7).standard_normal((nb, m, n))
        B = np.random.default_rng(8).standard_normal((nb, m, k))
        dA, dB = ctx.upload(A), ctx.upload(B)
        dX = ctx.alloc(nb * n * k * 8)
        dI = ctx.alloc(nb * 4)
        ctx.call("lq_lstsq_householder_batched_dev", dA.ptr, dB.ptr, nb, m, n, k, dX.ptr)
        ctx.sync()
        X = ctx.download(dX, (nb, n, k))
        Xo = orc.lstsq_householder_batched(A, B)
        e1 = orc.rel_max_err(X, Xo)
        ctx.call("lq_lstsq_mgs_batched_dev", dA.ptr, dB.ptr, nb, m, n, k, dX.ptr, dI.ptr)
        ctx.sync()
        X = ctx.download(dX, (nb, n, k))
        Xo = orc.lstsq_mgs_batched(A, B).reshape(nb, n, k)
        e2 = orc.rel_max_err(X, Xo)
        print("lstsq", (m, n, k), "hh", e1, "mgs", e2, flush=True)
        res[f"ls{m}x{n}x{k}"] = dict(hh=e1, mgs=e2)
    out["small"] = res


guarded(small_correct)


# ------------------------------------------------------------------ batched 32x32 timing
def hh32_time():
    section("hh32 timing (device resident, 2^18 matrices = 6.4 GB traffic, > L2)")
    nb = 1 << 18
    rng = np.random.default_rng(2)
    A = rng.standard_normal((nb, 32, 32))
    dA = ctx.upload(A)
    dQ = ctx.alloc(A.nbytes)
    dR = ctx.alloc(A.nbytes)
    dI = ctx.alloc(nb * 4)
    for reorth in (0, 1):
        for _ in range(2):
            ctx.call("lq_mgs_qr_batched_dev", dA.ptr, nb, 32, 32, reorth, dQ.ptr, dR.ptr, dI.ptr)
        ctx.sync()
        ts = []
        for _ in range(5):
            ctx.record(0)
            ctx.call("lq_mgs_qr_batched_dev", dA.ptr, nb, 32, 32, reorth, dQ.ptr, dR.ptr, dI.ptr)
            ctx.record(1)
            ts.append(ctx.elapsed_ms(0, 1))
        t = min(ts)
        out[f"mgs32_time_reorth{reorth}"] = dict(ms=t, mat_per_s=nb / t * 1e3, gbs=nb * 24576 / t / 1e6)
        print("mgs reorth", reorth, out[f"mgs32_time_reorth{reorth}"], flush=True)
    # host-pointer pipeline (pageable then pinned)
    Qh = np.empty_like(A)
    Rh = np.empty_like(A)
    t0 = time.perf_counter()
    ctx.call("lq_householder_qr_batched", A.ctypes.data, nb, 32, 32, Qh.ctypes.data, Rh.ctypes.data)
    t1 = time.perf_counter()
    print("e2e pageable: %.1f ms -> %.2f M mat/s" % ((t1 - t0) * 1e3, nb / (t1 - t0) / 1e6), flush=True)
    Ap = nat.pinned_empty(A.shape)
    Ap[...] = A
    Qp = nat.pinned_empty(A.shape)
    Rp = nat.pinned_empty(A.shape)
    for _ in range(2):
        t0 = time.perf_counter()
        ctx.call("lq_householder_qr_batched", Ap.ctypes.data, nb, 32, 32, Qp.ctypes.data, Rp.ctypes.data)
        t1 = time.perf_counter()
        print("e2e pinned: %.1f ms -> %.2f M mat/s" % ((t1 - t0) * 1e3, nb / (t1 - t0) / 1e6), flush=True)
    out["e2e_pinned_mat_per_s"] = nb / (t1 - t0)
    print("e2e check", orc.rel_max_err(Qp[:8], orc.householder_qr_batched(A[:8])[0]), flush=True)


guarded(hh32_time)

os.makedirs("gpurun_out", exist_ok=True)
with open("gpurun_out/check1.json", "w") as fh:
    json.dump(out, fh, indent=1, default=str)
print("\nDONE", flush=True)

#!/usr/bin/env python3
"""GPU bring-up 2: probes, GEMM, blocked Householder QR."""
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
what = set(sys.argv[1:]) or {"probes", "gemm", "blocked"}


def section(name):
    print(f"\n===== {name} =====", flush=True)


def guarded(fn):
    try:
        fn()
    except Exception:
        traceback.print_exc()
        sys.stdout.flush()


def probes():
    section("probes")
    print("dfma latency cycles", ctx.probe(4))
    names = ["rcp_seed", "rsqrt_seed", "rcp_nr3", "rsqrt_nr3", "sqrt_nr3", "rcp_nr2", "rsqrt_nr2"]
    for k, nme in enumerate(names):
        print(nme, "max rel err", ctx.probe(10 + k), flush=True)


def gemm_case(ta, tb, M, N, K, alpha=1.0, beta=0.0, reps=0):
    rng = np.random.default_rng(M + 3 * N + 7 * K)
    A = rng.standard_normal((K, M) if ta else (M, K))
    B = rng.standard_normal((N, K) if tb else (K, N))
    Cm = rng.standard_normal((M, N))
    dA, dB, dC = ctx.upload(A), ctx.upload(B), ctx.upload(Cm)
    ctx.call("lq_gemm_dev", int(ta), int(tb), M, N, K, alpha, dA.ptr, A.shape[1], dB.ptr, B.shape[1], beta, dC.ptr, N)
    ctx.sync()
    got = ctx.download(dC, (M, N))
    ref = alpha * ((A.T if ta else A) @ (B.T if tb else B)) + beta * Cm
    err = float(np.max(np.abs(got - ref)) / np.max(np.abs(ref)))
    msg = f"gemm ta={int(ta)} tb={int(tb)} M={M} N={N} K={K} a={alpha} b={beta}: rel err {err:.2e}"
    if reps:
        for _ in range(2):
            ctx.call("lq_gemm_dev", int(ta), int(tb), M, N, K, alpha, dA.ptr, A.shape[1], dB.ptr, B.shape[1], beta, dC.ptr, N)
        ctx.sync()
        ts = []
        for _ in range(reps):
            ctx.record(0)
            ctx.call("lq_gemm_dev", int(ta), int(tb), M, N, K, alpha, dA.ptr, A.shape[1], dB.ptr, B.shape[1], beta, dC.ptr, N)
            ctx.record(1)
            ts.append(ctx.elapsed_ms(0, 1))
        t = min(ts)
        msg += f"  {t:.3f} ms  {2.0*M*N*K/t/1e9:.2f} TFLOP/s"
    print(msg, flush=True)
    return err


def gemm():
    section("gemm correctness (fast + generic paths)")
    for ta in (False, True):
        for tb in (False, True):
            gemm_case(ta, tb, 128, 128, 64)
            gemm_case(ta, tb, 256, 384, 160, alpha=-1.0, beta=1.0)
            gemm_case(ta, tb, 200, 136, 48, alpha=0.5, beta=2.0)   # partial tiles
            gemm_case(ta, tb, 130, 70, 35)                          # K remainder, generic pieces
            gemm_case(ta, tb, 33, 17, 9)                            # generic only
    gemm_case(True, False, 32, 96, 4096)     # inner-panel W (split-K)
    gemm_case(True, False, 128, 2048, 8192)  # trailing W (split-K)
    gemm_case(False, False, 4096, 96, 32, alpha=-1.0, beta=1.0)
    section("gemm timing")
    gemm_case(False, False, 4096, 4096, 4096, reps=3)
    gemm_case(True, False, 4096, 4096, 4096, reps=3)
    gemm_case(False, False, 8192, 8192, 128, alpha=-1.0, beta=1.0, reps=3)   # rank-128 trailing update
    gemm_case(True, False, 128, 8192, 8192, reps=3)                            # W = V^T C
    gemm_case(True, False, 128, 128, 8192, reps=3)                             # Gram of a block
    gemm_case(False, False, 8192, 96, 32, alpha=-1.0, beta=1.0, reps=3)
    gemm_case(True, False, 32, 96, 8192, reps=3)


def blocked():
    section("blocked householder QR (single matrix)")
    print("max cluster before:", ctx.props()["max_cluster"])
    res = {}
    for (m, n) in [(64, 64), (100, 10), (96, 40), (130, 70), (256, 256), (300, 300), (512, 256), (700, 130), (1000, 1000), (2048, 512)]:
        A = np.random.default_rng(m * 7 + n).standard_normal((m, n))
        if (m, n) == (130, 70):
            A[:, 33] = 0.0  # skipped reflector inside a panel
        dA = ctx.upload(A)
        dQ = ctx.alloc(A.nbytes)
        dR = ctx.alloc(n * n * 8)
        t0 = time.perf_counter()
        ctx.call("lq_householder_qr_dev", dA.ptr, m, n, dQ.ptr, dR.ptr)
        ctx.sync()
        t1 = time.perf_counter()
        Q = ctx.download(dQ, (m, n))
        R = ctx.download(dR, (n, n))
        r = dict(resid=orc.qr_residual(A, Q, R), orth=orc.orth_error(Q), lower=float(np.max(np.abs(np.tril(R, -1)))) if n > 1 else 0.0)
        if m * n <= 1000 * 1000:
            Qo, Ro = orc.householder_qr(A)
            r["q"] = orc.rel_max_err(Q, Qo)
            r["r"] = orc.rel_max_err(R, Ro)
        else:
            Qn, Rn = np.linalg.qr(A)
            sg = np.sign(np.diag(Rn)) * np.sign(np.diag(R))
            r["r_vs_lapack_upto_sign"] = orc.rel_max_err(R * sg[:, None], Rn)
        r["first_call_ms"] = (t1 - t0) * 1e3
        print((m, n), r, flush=True)
        res[f"{m}x{n}"] = r
    print("max cluster after:", ctx.props()["max_cluster"])
    out["blocked"] = res
    section("blocked QR timing")
    for (m, n) in [(256, 256), (1024, 1024), (4096, 4096), (8192, 8192)]:
        A = np.random.default_rng(5).standard_normal((m, n))
        dA = ctx.upload(A)
        dQ = ctx.alloc(A.nbytes)
        dR = ctx.alloc(n * n * 8)
        ctx.call("lq_householder_qr_dev", dA.ptr, m, n, dQ.ptr, dR.ptr)
        ctx.sync()
        ts = []
        l0 = ctx.launches()
        for _ in range(3):
            ctx.record(0)
            ctx.call("lq_householder_qr_dev", dA.ptr, m, n, dQ.ptr, dR.ptr)
            ctx.record(1)
            ts.append(ctx.elapsed_ms(0, 1))
        t = min(ts)
        flops = 2 * (2.0 * m * n * n - 2.0 / 3.0 * n ** 3)
        print(f"{m}x{n}: {t:.2f} ms  F_QR {flops/t/1e9:.2f} TFLOP/s  launches/call {(ctx.launches()-l0)//3}", flush=True)
        out[f"blocked_time_{m}"] = dict(ms=t, tflops=flops / t / 1e9)
        if m == 8192:
            Q = ctx.download(dQ, (m, n))
            R = ctx.download(dR, (n, n))
            print("8192 resid", orc.qr_residual(A, Q, R), "orth", orc.orth_error(Q[:, :512]), flush=True)


for name in ("probes", "gemm", "blocked"):
    if name in what:
        guarded(globals()[name])

os.makedirs("gpurun_out", exist_ok=True)
with open("gpurun_out/check2.json", "w") as fh:
    json.dump(out, fh, indent=1, default=str)
print("\nDONE", flush=True)

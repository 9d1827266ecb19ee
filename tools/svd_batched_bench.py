#!/usr/bin/env python3
"""Batched economy SVD (svd_batched), device resident, against the ways the library and the host computed it before.

Arms:
  kernel      lq_svd_gram_batched_dev on 2^20 x 32 x 32 and 2^16 x 256 x 16 (8 GiB and 4 GiB of input, both larger than
              the 126 MB L2), CUDA events around each call after warm-ups, min and median of the repetitions
  loop        lq_svd_gram_dev (the single-matrix pipeline, which reads the rank back to the host) on 1024 matrices of the
              same shape, host clock around the loop
  m_small     the kernel and the loop at m = 4096, n = 32 (the tallest kernel shape, SvdSmall::M_SMALL), 1024 matrices
  numpy       np.linalg.svd of a stacked batch (2^16 x 32 x 32, 2^14 x 256 x 16) on the host cores
  host_ptr    lq_svd_gram_batched with pinned host buffers, 2^18 x 32 x 32, against bare copies of the same bytes (the host
              copy ceiling of DESIGN.md section 4-v)
Rates: matrices/s; bytes/s against the 6552 GB/s device copy peak (A read once, U, s, Vt and the rank written once); the
FP64 share against the 36.7 TFLOP/s DFMA peak, from 4 m n^2 flops (Gram and U) + 18 n flops per rotation, with the
rotations and sweeps per matrix counted by a host replica of the kernel's Jacobi on 64 of the input matrices.  The kernel's
singular values must agree with the loop's to 1e-12 (relative to s_1) before anything is printed.  The card's name and
power limit are printed with the numbers.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from linalg_b200 import _native as nat  # noqa: E402

COPY_PEAK = 6552e9
DFMA_PEAK = 36.7e12


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines() if q.returncode == 0 else ["unknown"]


def timed(ctx, fn, warmup, reps):
    for _ in range(warmup):
        fn()
    ms = []
    for _ in range(reps):
        ctx.record(0)
        fn()
        ctx.record(1)
        ctx.sync()
        ms.append(ctx.elapsed_ms(0, 1))
    return min(ms), float(np.median(ms))


def rr_pair(ne, rd, k):
    mod = ne - 1
    a, b = (ne - 1, rd % mod) if k == 0 else ((rd + k) % mod, (rd - k + mod) % mod)
    return min(a, b), max(a, b)


def jacobi_work(A):
    """(sweeps, rotations) of the kernel's two-sided Jacobi on A^T A: same scaling, order and rotation test."""
    G = A.T @ A
    n = G.shape[0]
    ne = n + (n & 1)
    Gp = np.zeros((ne, ne))
    Gp[:n, :n] = G
    d = np.max(np.abs(np.diag(G)))
    e = int(np.floor(np.log2(d))) if d > 0 else 0
    Gp = np.ldexp(Gp, -e)
    floor_abs, rel = 4.9303806576313238e-32 * np.ldexp(d, -e), 4 * 1.1102230246251565e-16
    rotations = 0
    for sweep in range(40):
        rotated = False
        for rd in range(ne - 1):
            pairs = [rr_pair(ne, rd, k) for k in range(ne // 2)]
            J = np.eye(ne)
            for p, q in pairs:
                app, aqq, apq = Gp[p, p], Gp[q, q], Gp[p, q]
                if abs(apq) > floor_abs and abs(apq) > rel * np.sqrt(abs(app * aqq)):
                    tau = (aqq - app) / (2 * apq)
                    t = np.copysign(1.0, tau) / (abs(tau) + np.sqrt(1 + tau * tau))
                    c = 1 / np.sqrt(1 + t * t)
                    s = t * c
                    J[p, p], J[q, q], J[p, q], J[q, p] = c, c, s, -s
                    rotated = True
                    rotations += 1
            Gp = J.T @ Gp @ J
        if not rotated:
            return sweep + 1, rotations
    return 40, rotations


def device_batch(ctx, b, m, n, seed):
    bufs = dict(A=ctx.alloc(8 * b * m * n), U=ctx.alloc(8 * b * m * n), s=ctx.alloc(8 * b * n), Vt=ctx.alloc(8 * b * n * n),
                r=ctx.alloc(4 * b))
    ctx.call("lq_random_normal_dev", bufs["A"].ptr, b * m * n, seed)
    return bufs


def kernel_call(ctx, d, b, m, n):
    return lambda: ctx.call("lq_svd_gram_batched_dev", d["A"].ptr, b, m, n, 1e-12, d["U"].ptr, d["s"].ptr, d["Vt"].ptr, d["r"].ptr)


def loop_time(ctx, d, cnt, m, n):
    """Seconds per matrix of lq_svd_gram_dev over the first cnt matrices of d; their s go to sl (host)."""
    rank = C.c_int(0)
    dU, ds, dV = ctx.alloc(8 * m * n), ctx.alloc(8 * n), ctx.alloc(8 * n * n)
    sl = np.empty((cnt, n))

    def one(i):
        ctx.call("lq_svd_gram_dev", d["A"].ptr + 8 * i * m * n, m, n, 1e-12, dU.ptr, ds.ptr, dV.ptr, C.byref(rank))

    for i in range(8):
        one(i)
    ctx.sync()
    t0 = time.perf_counter()
    for i in range(cnt):
        one(i)
    ctx.sync()
    dt = (time.perf_counter() - t0) / cnt
    for i in range(cnt):
        one(i)
        sl[i] = ctx.download(ds, (n,))
    return dt, sl


def sample(ctx, buf, i, shape):
    out = np.empty(shape)
    ctx.call("lq_memcpy_d2h", out.ctypes.data, buf.ptr + out.nbytes * i, out.nbytes)
    ctx.sync()
    return out


def shape_arm(ctx, b, m, n, loop_cnt, np_cnt, warmup, reps):
    d = device_batch(ctx, b, m, n, 7 + n)
    tmin, tmed = timed(ctx, kernel_call(ctx, d, b, m, n), warmup, reps)
    s = ctx.download(d["s"], (b, n))
    dt_loop, sl = loop_time(ctx, d, loop_cnt, m, n)
    s_diff = float(np.max(np.abs(s[:loop_cnt] - sl) / sl[:, :1]))
    assert s_diff <= 1e-12, s_diff
    work = [jacobi_work(sample(ctx, d["A"], i, (m, n))) for i in range(64)]
    sweeps = float(np.mean([w[0] for w in work]))
    rots = float(np.mean([w[1] for w in work]))
    flops = 4.0 * m * n * n + 18.0 * n * rots
    nbytes = 8.0 * (2 * m * n + n * n + n) + 4
    sec = tmin * 1e-3
    A_host = np.random.default_rng(1).standard_normal((np_cnt, m, n))
    t0 = time.perf_counter()
    np.linalg.svd(A_host, full_matrices=False)
    t_np = (time.perf_counter() - t0) / np_cnt
    del d
    return {
        "shape": [b, m, n], "kernel_ms_min": tmin, "kernel_ms_median": tmed, "matrices_per_s": b / sec,
        "bytes_per_s": b * nbytes / sec, "copy_peak_share": b * nbytes / sec / COPY_PEAK,
        "sweeps_mean": sweeps, "rotations_mean": rots, "flops_per_matrix": flops,
        "fp64_share": b * flops / sec / DFMA_PEAK,
        "loop_us_per_matrix": dt_loop * 1e6, "loop_matrices": loop_cnt, "speedup_vs_loop": dt_loop * b / sec,
        "s_max_rel_diff_vs_loop": s_diff,
        "numpy_us_per_matrix": t_np * 1e6, "numpy_matrices": np_cnt,
    }


def m_small_arm(ctx, warmup, reps):
    b, m, n = 1024, 4096, 32
    d = device_batch(ctx, b, m, n, 11)
    tmin, _ = timed(ctx, kernel_call(ctx, d, b, m, n), warmup, reps)
    dt_loop, _ = loop_time(ctx, d, 64, m, n)
    return {"shape": [b, m, n], "kernel_us_per_matrix": tmin * 1e3 / b, "loop_us_per_matrix": dt_loop * 1e6, "loop_matrices": 64}


def host_ptr_arm(ctx, warmup, reps):
    b, m, n = 1 << 18, 32, 32
    A = nat.pinned_empty((b, m, n))
    A[...] = np.random.default_rng(3).standard_normal((b, m, n))
    U, s, Vt, r = nat.pinned_empty((b, m, n)), nat.pinned_empty((b, n)), nat.pinned_empty((b, n, n)), nat.pinned_empty((b,), np.int32)

    def run():
        ctx.call("lq_svd_gram_batched", A.ctypes.data, b, m, n, 1e-12, U.ctypes.data, s.ctypes.data, Vt.ctypes.data, r.ctypes.data)

    for _ in range(warmup):
        run()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        run()
        ts.append(time.perf_counter() - t0)
    dA, dO = ctx.alloc(A.nbytes), ctx.alloc(U.nbytes + Vt.nbytes + s.nbytes)

    def copies():
        ctx.call("lq_memcpy_h2d", dA.ptr, A.ctypes.data, A.nbytes)
        ctx.call("lq_memcpy_d2h", U.ctypes.data, dO.ptr, U.nbytes)
        ctx.call("lq_memcpy_d2h", Vt.ctypes.data, dO.ptr + U.nbytes, Vt.nbytes)
        ctx.call("lq_memcpy_d2h", s.ctypes.data, dO.ptr + U.nbytes + Vt.nbytes, s.nbytes)
        ctx.sync()

    copies()
    tc = []
    for _ in range(reps):
        t0 = time.perf_counter()
        copies()
        tc.append(time.perf_counter() - t0)
    return {"shape": [b, m, n], "host_ptr_ms": min(ts) * 1e3, "matrices_per_s": b / min(ts),
            "bare_copies_ms": min(tc) * 1e3, "copy_bound_share": min(tc) / min(ts)}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the JSON result here")
    a = ap.parse_args()
    ctx = nat.Context(0)
    res = {
        "card": card(),
        "host_cores": os.cpu_count(),
        "blas_threads": os.environ.get("OMP_NUM_THREADS", "library default"),
        "arms": [shape_arm(ctx, 1 << 20, 32, 32, 1024, 1 << 16, a.warmup, a.reps),
                 shape_arm(ctx, 1 << 16, 256, 16, 1024, 1 << 14, a.warmup, a.reps)],
        "m_small": m_small_arm(ctx, a.warmup, a.reps),
        "host_ptr": host_ptr_arm(ctx, a.warmup, a.reps),
    }
    try:
        from threadpoolctl import threadpool_info

        res["blas_threads"] = [(i.get("internal_api"), i.get("num_threads")) for i in threadpool_info()]
    except ImportError:
        pass
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()

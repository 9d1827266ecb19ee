#!/usr/bin/env python3
"""Tall-skinny least squares, device resident: lq_lstsq_tsqr_dev against the two ways the library solved the same system
before it existed.

Arms, on the same 2^20 x 128 A (1 GiB, larger than the 126 MB L2) with 16 right-hand sides:
  lstsq_tsqr    lq_lstsq_tsqr_dev (CholeskyQR2, pass 2 as one fused [Q1 | B] sweep, Q never formed)
  householder   lq_lstsq_householder_batched_info_dev with batch 1 (the blocked Householder route)
  composition   lq_tsqr_dev, then Q^T B with lq_gemm_dev; the n x n triangular solve R X = Q^T B runs on the host and is
                not timed (so this arm is a lower bound of the composition)
The arms must agree to 1e-10 (max relative difference of X) before anything is printed.  Times are CUDA events around each
call after warm-ups, min and median of the repetitions.  GFLOP/s on two counts:
  algorithmic: F_R + 4 m n k with F_R = 2 m n^2 - 2 n^3 / 3 (Householder R);  executed: 4 m n^2 + 2 m n k (CholeskyQR2).
With two or more GPUs it also times lq_lstsq_tsqr_sharded_dev on 8M x 128 split over all of them (one process per GPU).
The card's name and power limit are printed with the numbers.
"""
import argparse
import ctypes as C
import json
import os
import socket
import subprocess
import sys

import numpy as np
from scipy.linalg import solve_triangular

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from linalg_b200 import _native as nat  # noqa: E402


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
        ms.append(ctx.elapsed_ms(0, 1))
    return min(ms), float(np.median(ms))


def flops(m, n, k):
    alg = 2.0 * m * n * n - 2.0 * n ** 3 / 3.0 + 4.0 * m * n * k
    exe = 4.0 * m * n * n + 2.0 * m * n * k
    return alg, exe


def one_gpu(m, n, k, warmup, reps):
    ctx = nat.Context(0)
    dA = ctx.alloc(8 * m * n)
    dB = ctx.alloc(8 * m * k)
    ctx.call("lq_random_normal_dev", dA.ptr, m * n, 1)
    ctx.call("lq_random_normal_dev", dB.ptr, m * k, 2)
    dX = {a: ctx.alloc(8 * n * k) for a in ("lstsq_tsqr", "householder", "composition")}
    dI, dQ, dR, dY = ctx.alloc(16), ctx.alloc(8 * m * n), ctx.alloc(8 * n * n), ctx.alloc(8 * n * k)
    arms = {
        "lstsq_tsqr": lambda: ctx.call("lq_lstsq_tsqr_dev", dA.ptr, m, n, dB.ptr, k, dX["lstsq_tsqr"].ptr, dI.ptr),
        "householder": lambda: ctx.call("lq_lstsq_householder_batched_info_dev", dA.ptr, dB.ptr, 1, int(m), n, k,
                                        dX["householder"].ptr, dI.ptr),
        "composition": lambda: (ctx.call("lq_tsqr_dev", dA.ptr, m, n, dQ.ptr, dR.ptr),
                                ctx.call("lq_gemm_dev", 1, 0, n, k, int(m), C.c_double(1.0), dQ.ptr, n, dB.ptr, k,
                                         C.c_double(0.0), dY.ptr, k)),
    }
    res = {}
    for name, fn in arms.items():
        res[name] = timed(ctx, fn, warmup, reps)
    X = {name: ctx.download(dX[name], (n, k)) for name in ("lstsq_tsqr", "householder")}
    X["composition"] = solve_triangular(ctx.download(dR, (n, n)), ctx.download(dY, (n, k)))
    ref = X["householder"]
    for name, x in X.items():
        d = float(np.max(np.abs(x - ref)) / np.max(np.abs(ref)))
        assert d <= 1e-10, (name, d)
    alg, exe = flops(m, n, k)
    out = {"card": card(), "shape": [m, n, k], "warmup": warmup, "reps": reps}
    for name, (mn, md) in res.items():
        out[name] = {"ms_min": round(mn, 3), "ms_median": round(md, 3), "alg_gflops": round(alg / mn / 1e6, 1),
                     "exec_gflops": round(exe / mn / 1e6, 1)}
    return out


def _worker(rank, world, port, m, n, k, warmup, reps, outdir):
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1",
                      MASTER_PORT=str(port), LINALG_B200_DEVICE=str(rank))
    import linalg_b200 as lb
    from linalg_b200 import dist as d
    from linalg_b200.utils import shard_bounds

    info = d.init_control_plane("gloo")
    ctx = lb.Context(rank)
    d.init_comm(ctx, info)
    lo, hi = shard_bounds(m, world, rank)
    dA, dB = ctx.alloc(8 * (hi - lo) * n), ctx.alloc(8 * (hi - lo) * k)
    ctx.call("lq_random_normal_dev", dA.ptr, (hi - lo) * n, 10 + rank)
    ctx.call("lq_random_normal_dev", dB.ptr, (hi - lo) * k, 20 + rank)
    dX, dI = ctx.alloc(8 * n * k), ctx.alloc(16)
    fn = lambda: ctx.call("lq_lstsq_tsqr_sharded_dev", dA.ptr, hi - lo, n, dB.ptr, k, dX.ptr, dI.ptr)  # noqa: E731
    mn, md = timed(ctx, fn, warmup, reps)
    np.savez(os.path.join(outdir, f"r{rank}.npz"), ms=[mn, md], X=ctx.download(dX, (n, k)))
    d.barrier()
    ctx.call("lq_comm_destroy")
    d.shutdown_control_plane()


def sharded(world, m, n, k, warmup, reps):
    import tempfile

    import torch.multiprocessing as mp

    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    with tempfile.TemporaryDirectory() as tmp:
        mp.spawn(_worker, args=(world, port, m, n, k, warmup, reps, tmp), nprocs=world, join=True)
        z = [np.load(os.path.join(tmp, f"r{r}.npz")) for r in range(world)]
        assert all(np.array_equal(z[0]["X"], q["X"]) for q in z), "X not replicated"
        ms = max(q["ms"][0] for q in z), max(q["ms"][1] for q in z)
    alg, exe = flops(m, n, k)
    return {"card": card(), "gpus": world, "shape": [m, n, k], "ms_min": round(ms[0], 3), "ms_median": round(ms[1], 3),
            "alg_gflops": round(alg / ms[0] / 1e6, 1), "exec_gflops": round(exe / ms[0] / 1e6, 1)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--m", type=int, default=1 << 20)
    ap.add_argument("--n", type=int, default=128)
    ap.add_argument("--k", type=int, default=16)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--sharded-m", type=int, default=8 << 20)
    a = ap.parse_args()
    print(json.dumps({"one_gpu": one_gpu(a.m, a.n, a.k, a.warmup, a.reps)}), flush=True)
    world = nat.device_count()
    if world >= 2:
        print(json.dumps({"sharded": sharded(world, a.sharded_m, a.n, a.k, a.warmup, a.reps)}), flush=True)
    else:
        print(json.dumps({"sharded": f"skipped: {world} GPU"}), flush=True)


if __name__ == "__main__":
    main()

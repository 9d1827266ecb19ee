#!/usr/bin/env python3
"""Race-detection substitute (compute-sanitizer is closed on this pool): every kernel family is run REPS times on the same
device-resident input and the outputs must be bitwise identical (SHA-1 of the raw bytes) -- shared-memory / shuffle / DSMEM /
st.async races typically show up as run-to-run differences.  python tools/soak_determinism.py [reps=25]"""
import ctypes as C, hashlib, os, sys
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from linalg_b200 import _native as nat
REPS = int(sys.argv[1]) if len(sys.argv) > 1 else 25
ctx = nat.Context(0)
rng = np.random.default_rng(99)

def digest(*bufs_shapes):
    h = hashlib.sha1()
    for buf, shape, dt in bufs_shapes:
        h.update(ctx.download(buf, shape, dtype=dt).tobytes())
    return h.hexdigest()

def soak(name, run, outs):
    seen = set()
    for _ in range(REPS):
        for buf, shape, dt in outs:
            ctx.call("lq_memset", buf.ptr, 0xA5, int(np.prod(shape)) * np.dtype(dt).itemsize)
        run()
        seen.add(digest(*outs))
    print(f"{name:42s} {REPS} runs -> {len(seen)} distinct result(s)", flush=True)
    assert len(seen) == 1, name

nb = 40003
A = rng.standard_normal((nb, 32, 32)); dA = ctx.upload(A); dQ, dR, dI = ctx.alloc(A.nbytes), ctx.alloc(A.nbytes), ctx.alloc(4 * nb)
soak("householder_qr_batched 32x32 (c8 kernel)", lambda: ctx.call("lq_householder_qr_batched_dev", dA.ptr, nb, 32, 32, dQ.ptr, dR.ptr, 0),
     [(dQ, (nb, 32, 32), np.float64), (dR, (nb, 32, 32), np.float64)])
for re in (0, 1):
    soak(f"qr_batched 32x32 (MGS, reorth={re})", lambda: ctx.call("lq_mgs_qr_batched_dev", dA.ptr, nb, 32, 32, re, dQ.ptr, dR.ptr, dI.ptr),
         [(dQ, (nb, 32, 32), np.float64), (dR, (nb, 32, 32), np.float64), (dI, (nb,), np.int32)])
ns = 3001
A3 = rng.standard_normal((ns, 256, 64)); B3 = rng.standard_normal((ns, 256, 16))
d3, dB3, dX = ctx.upload(A3), ctx.upload(B3), ctx.alloc(8 * ns * 64 * 16)
soak("least squares 256x64x16 (tile kernel)", lambda: ctx.call("lq_lstsq_householder_batched_dev", d3.ptr, dB3.ptr, ns, 256, 64, 16, dX.ptr),
     [(dX, (ns, 64, 16), np.float64)])
A4 = rng.standard_normal((700, 97, 23)); B4 = rng.standard_normal((700, 97, 5))
d4, dB4, dX4 = ctx.upload(A4), ctx.upload(B4), ctx.alloc(8 * 700 * 23 * 5)
soak("least squares 97x23x5 (ragged tile kernel)", lambda: ctx.call("lq_lstsq_householder_batched_dev", d4.ptr, dB4.ptr, 700, 97, 23, 5, dX4.ptr),
     [(dX4, (700, 23, 5), np.float64)])
m, n = 300017, 128
A5 = rng.standard_normal((m, n)); d5 = ctx.upload(A5); dG = ctx.alloc(8 * n * n)
dQ5, dR5, ds, dVt = ctx.alloc(A5.nbytes), ctx.alloc(8 * n * n), ctx.alloc(8 * n), ctx.alloc(8 * n * n)
soak("gram 300017x128 (SYRK, split over 148 CTAs)", lambda: ctx.call("lq_gram_dev", d5.ptr, m, n, dG.ptr), [(dG, (n, n), np.float64)])
soak("tsqr 300017x128 (CholeskyQR2)", lambda: ctx.call("lq_tsqr_dev", d5.ptr, m, n, dQ5.ptr, dR5.ptr),
     [(dQ5, (m, n), np.float64), (dR5, (n, n), np.float64)])
soak("svd 300017x128 (Gram + Jacobi)", lambda: ctx.call("lq_svd_gram_dev", d5.ptr, m, n, C.c_double(1e-12), dQ5.ptr, ds.ptr, dVt.ptr, C.byref(C.c_int(0))),
     [(dQ5, (m, n), np.float64), (ds, (n,), np.float64), (dVt, (n, n), np.float64)])
for nn in (256, 1000, 2500):
    A6 = rng.standard_normal((nn, nn)); d6 = ctx.upload(A6); dQ6, dR6 = ctx.alloc(A6.nbytes), ctx.alloc(A6.nbytes)
    soak(f"householder_qr {nn}^2 (blocked, graph replay)", lambda: ctx.call("lq_householder_qr_dev", d6.ptr, nn, nn, dQ6.ptr, dR6.ptr),
         [(dQ6, (nn, nn), np.float64), (dR6, (nn, nn), np.float64)])
    for b in (d6, dQ6, dR6):
        b.free()
print("all deterministic")

#!/usr/bin/env python3
"""Tiny driver for ncu: run the batched 32x32 kernels a few times on device-resident data.

usage: python tools/prof_batched.py [log2_batch=16] [mgs=0]
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from linalg_b200 import _native as nat  # noqa: E402

lg = int(sys.argv[1]) if len(sys.argv) > 1 else 16
mgs = int(sys.argv[2]) if len(sys.argv) > 2 else 0
reps = int(os.environ.get('PROF_REPS', '3'))
nb = 1 << lg
ctx = nat.Context(0)
A = np.random.default_rng(2).standard_normal((nb, 32, 32))
dA = ctx.upload(A)
dQ = ctx.alloc(A.nbytes)
dR = ctx.alloc(A.nbytes)
dI = ctx.alloc(nb * 4)
for _ in range(reps):
    ctx.record(0)
    ctx.call("lq_householder_qr_batched_dev", dA.ptr, nb, 32, 32, dQ.ptr, dR.ptr, 0)
    ctx.record(1)
    ms = ctx.elapsed_ms(0, 1)
print(f"householder: {ms:.3f} ms  {nb/ms/1e3:.1f} M mat/s")
if mgs:
    for _ in range(reps):
        ctx.record(0)
        ctx.call("lq_mgs_qr_batched_dev", dA.ptr, nb, 32, 32, 0, dQ.ptr, dR.ptr, dI.ptr)
        ctx.record(1)
        ms = ctx.elapsed_ms(0, 1)
    print(f"mgs: {ms:.3f} ms  {nb/ms/1e3:.1f} M mat/s")
ctx.sync()

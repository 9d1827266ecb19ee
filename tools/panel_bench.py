#!/usr/bin/env python3
"""Panel kernels of the blocked QR (K4a): agreement between the versions + time per launch."""
import os, sys
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from linalg_b200 import _native as nat
ctx = nat.Context(0)
LDA = 8192
def run(A, version, reps=0):
    m = A.shape[0]
    buf = np.zeros((m, LDA)); buf[:, :32] = A
    dA = ctx.upload(buf); dV = ctx.upload(np.zeros((m, LDA))); dT = ctx.upload(np.zeros((32, 128)))
    ctx.call("lq_debug_panel", dA.ptr, LDA, dV.ptr, LDA, dT.ptr, 128, m, 32, version)
    R = ctx.download(dA, (m, LDA))[:32, :32].copy(); V = ctx.download(dV, (m, LDA))[:, :32].copy()
    T = ctx.download(dT, (32, 128))[:, :32].copy()
    t = None
    if reps:
        for _ in range(3): ctx.call("lq_debug_panel", dA.ptr, LDA, dV.ptr, LDA, dT.ptr, 128, m, 32, version)
        ctx.record(0)
        for _ in range(reps): ctx.call("lq_debug_panel", dA.ptr, LDA, dV.ptr, LDA, dT.ptr, 128, m, 32, version)
        ctx.record(1)
        t = ctx.elapsed_ms(0, 1) / reps * 1e3
    for b in (dA, dV, dT): b.free()
    return np.triu(R), V, T, t
def rel(a, b): return float(np.max(np.abs(a - b)) / max(1e-300, np.max(np.abs(b))))
for m in (8192, 5000, 4096, 2048, 1000, 512, 300, 256, 200, 64, 33, 32):
    A = np.random.default_rng(m).standard_normal((m, 32))
    if m in (300, 200): A[:, 7] = 0.0; A[:, 20] = A[:, 3]   # a skipped reflector and a dependent column
    Qn, Rn = np.linalg.qr(A)
    ref = run(A, 1, 20)
    line = f"m={m:5d} v1 {ref[3]:7.1f} us"
    for ver in (3, 0):
        if ver == 0 and m > 256: continue   # version 0 = default: the one-CTA SOLO kernel up to 256 rows
        if ver == 3 and m > 16 * 256: continue
        got = run(A, ver, 20)
        # invariants: (I - V T V^T)^T A = [R; 0]
        QtA = A - got[1] @ (got[2].T @ (got[1].T @ A))
        inv = float(np.max(np.abs(QtA[:32] - got[0])) / np.max(np.abs(A))), float(np.max(np.abs(QtA[32:])) if m > 32 else 0.0)
        line += f" | v{ver} {got[3]:7.1f} us dR {rel(got[0], ref[0]):.1e} dV {rel(got[1], ref[1]):.1e} dT {rel(got[2], ref[2]):.1e} inv {inv[0]:.1e} {inv[1]:.1e}"
    print(line, flush=True)

"""In-tree build of liblinalg_b200.so with nvcc for sm_100a (no torch, no cmake).

``python -m linalg_b200.build`` or ``linalg_b200.build.build()``.  Objects go to
``linalg_b200/csrc/build/`` and the library to ``linalg_b200/_lib/`` (both git-ignored;
the library travels to the GPU box with the tree).
"""
from __future__ import annotations

import concurrent.futures as cf
import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(CSRC, "build")
LIBDIR = os.path.join(HERE, "_lib")
LIB = os.path.join(LIBDIR, "liblinalg_b200.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC,-O2",
    "--expt-relaxed-constexpr",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; linalg_b200 cannot be built (there is no CPU fallback)")


def _sources():
    return sorted(f for f in os.listdir(CSRC) if f.endswith(".cu"))


def _headers_digest() -> str:
    h = hashlib.sha1()
    for root in (CSRC, os.path.join(HERE, "..", "include")):
        for f in sorted(os.listdir(root)):
            if f.endswith((".cuh", ".h")):
                with open(os.path.join(root, f), "rb") as fh:
                    h.update(fh.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False, ptxas_info: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    os.makedirs(LIBDIR, exist_ok=True)
    nvcc = _nvcc()
    digest = _headers_digest()
    stamp = os.path.join(OBJ, "headers.sha1")
    old = open(stamp).read() if os.path.exists(stamp) else ""
    hdr_changed = old != digest

    jobs = []
    for src in _sources():
        s = os.path.join(CSRC, src)
        o = os.path.join(OBJ, src[:-3] + ".o")
        if force or hdr_changed or not os.path.exists(o) or os.path.getmtime(o) < os.path.getmtime(s):
            cmd = [nvcc, *NVCC_FLAGS, "-I", CSRC, "-c", s, "-o", o]
            if ptxas_info:
                cmd[1:1] = ["-Xptxas", "-v"]
            jobs.append((src, cmd))

    def run(job):
        src, cmd = job
        p = subprocess.run(cmd, capture_output=True, text=True)
        return src, p.returncode, p.stdout + p.stderr

    failed = False
    if jobs:
        with cf.ThreadPoolExecutor(max_workers=min(8, len(jobs))) as ex:
            for src, rc, out in ex.map(run, jobs):
                if verbose or rc != 0 or ptxas_info:
                    sys.stderr.write(f"--- nvcc {src} (rc={rc})\n{out}\n")
                failed |= rc != 0
    if failed:
        raise RuntimeError("nvcc failed, see output above")
    objs = [os.path.join(OBJ, s[:-3] + ".o") for s in _sources()]
    if jobs or not os.path.exists(LIB):
        cmd = [nvcc, "-shared", "-o", LIB, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC",
               "-lcudart_static", "-ldl", "-lpthread", "-lrt"]
        p = subprocess.run(cmd, capture_output=True, text=True)
        if p.returncode != 0:
            raise RuntimeError("link failed:\n" + p.stdout + p.stderr)
    with open(stamp, "w") as fh:
        fh.write(digest)
    return LIB


if __name__ == "__main__":
    path = build(force="--force" in sys.argv, verbose="-v" in sys.argv, ptxas_info="--ptxas" in sys.argv)
    print(path)

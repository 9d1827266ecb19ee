"""Host-side logic that needs no GPU: argument checking of the drop-in API, sharding arithmetic,
and the multi-rank control plane on gloo (world_size 2)."""
import os
import socket
import sys

import numpy as np
import pytest

import linalg_b200 as lb
from linalg_b200 import dist as lbdist
from linalg_b200.utils import as_f64_batch, as_f64_matrix, shard_bounds
from oracle import linalg_oracle as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_public_names_mirror_reference():
    # reference linalg/__init__.py:65-96 (hot-path names) + EPS from linalg/utils.py:9
    for name in ("qr", "householder_qr", "least_squares_qr", "least_squares_householder_qr", "svd",
                 "random_nonsingular_qr", "EPS"):
        assert hasattr(lb, name), name
    assert lb.EPS == 1e-12 == orc.EPS


def test_shape_errors_are_value_errors_before_any_device_work():
    with pytest.raises(ValueError):
        lb.householder_qr(np.ones(3))  # ndim != 2 (qr.py:71 tuple unpack)
    with pytest.raises(ValueError):
        lb.householder_qr(np.ones((2, 3)))  # m < n (matmul mismatch upstream)
    with pytest.raises(ValueError):
        lb.qr(np.ones((2, 2, 2)))
    with pytest.raises(ValueError):
        lb.householder_qr_batched(np.ones((4, 4)))
    with pytest.raises(ValueError):
        lb.least_squares_householder_qr(np.ones((2, 3)), np.ones(2))
    with pytest.raises(ValueError):
        lb.least_squares_householder_qr_batched(np.ones((2, 8, 4)), np.ones((3, 8, 1)))
    with pytest.raises(ValueError):
        lb.svd(np.ones(5))
    with pytest.raises(ValueError):
        lb.tsqr(np.ones((3, 5)))


def test_input_conversion_never_aliases_or_mutates():
    A = np.arange(12, dtype=np.int32).reshape(4, 3)
    W = as_f64_matrix(A)
    assert W.dtype == np.float64 and W.flags.c_contiguous and not np.shares_memory(W, A)
    F = np.asfortranarray(np.random.default_rng(0).standard_normal((5, 4)))
    W = as_f64_matrix(F)
    assert W.flags.c_contiguous and np.array_equal(W, F)
    assert as_f64_batch(np.zeros((2, 3, 3), dtype=np.float32)).dtype == np.float64


@pytest.mark.parametrize("total,n", [(1 << 20, 1), (1 << 20, 2), (1 << 20, 8), (1000, 3), (7, 8), (0, 4), (65536, 4)])
def test_shard_bounds_partition(total, n):
    spans = [shard_bounds(total, n, r) for r in range(n)]
    assert spans[0][0] == 0 and spans[-1][1] == total
    for (a0, a1), (b0, b1) in zip(spans, spans[1:]):
        assert a1 == b0 and a0 <= a1 and b0 <= b1
    sizes = [b - a for a, b in spans]
    assert max(sizes) - min(sizes) <= 1


def test_shard_bounds_alignment_and_errors():
    spans = [shard_bounds(1000, 3, r, align=64) for r in range(3)]
    assert spans[-1][1] == 1000 and all(a % 64 == 0 for a, _ in spans)
    with pytest.raises(ValueError):
        shard_bounds(10, 0, 0)
    with pytest.raises(ValueError):
        shard_bounds(10, 2, 2)


def test_row_sharded_math_single_process():
    """The exchange steps of SURVEY.md 8e are exact: sum of shard Grams = Gram; R of stacked shard R's = R."""
    A = np.random.default_rng(6).standard_normal((4096, 32))
    parts = [A[slice(*shard_bounds(4096, 4, r))] for r in range(4)]
    G = sum(p.T @ p for p in parts)
    assert orc.rel_max_err(G, A.T @ A) < 1e-13
    Rs = np.vstack([orc.tsqr_reference(p)[1] for p in parts])
    _, R = orc.tsqr_reference(Rs)
    assert orc.rel_max_err(R, orc.tsqr_reference(A)[1]) < 1e-12


# ------------------------------------------------------------------ gloo, world_size 2
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, outdir):
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1",
                      MASTER_PORT=str(port))
    sys.path.insert(0, ROOT)
    import torch.distributed as dist

    from linalg_b200 import dist as d
    from oracle import linalg_oracle as o

    info = d.init_control_plane("gloo")
    assert (info.rank, info.world) == (rank, world)
    # unique-id hand-off (128 bytes from rank 0)
    ident = bytes(range(128)) if rank == 0 else None
    got = d.broadcast_bytes(ident, 128)
    assert got == bytes(range(128))
    # timing reduction used by bench.py
    assert d.max_over_ranks(1.0 + rank) == float(world)
    assert d.sum_over_ranks(1.0) == float(world)
    # batch-sharded path: every rank factors its slice, no communication, union == whole batch
    A = np.random.default_rng(2).standard_normal((10, 8, 8))
    lo, hi = d.my_batch_slice(10, info)
    Q, R = o.householder_qr_batched(A[lo:hi])
    np.savez(os.path.join(outdir, f"r{rank}.npz"), lo=lo, hi=hi, Q=Q, R=R)
    # row-sharded path: Gram all-reduce gives the same G on every rank
    import torch

    T = np.random.default_rng(6).standard_normal((1000, 16))
    r0, r1 = d.my_row_slice(1000, info)
    g = torch.from_numpy(T[r0:r1].T @ T[r0:r1])
    dist.all_reduce(g)
    assert o.rel_max_err(g.numpy(), T.T @ T) < 1e-13
    d.barrier()
    d.shutdown_control_plane()


def test_control_plane_gloo_world2(tmp_path):
    import torch.multiprocessing as mp

    port = _free_port()
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    A = np.random.default_rng(2).standard_normal((10, 8, 8))
    Qo, Ro = orc.householder_qr_batched(A)
    seen = np.zeros(10, dtype=bool)
    for r in range(2):
        z = np.load(tmp_path / f"r{r}.npz")
        lo, hi = int(z["lo"]), int(z["hi"])
        assert np.array_equal(z["Q"], Qo[lo:hi]) and np.array_equal(z["R"], Ro[lo:hi])
        seen[lo:hi] = True
    assert seen.all()


def test_fan_out_splits_contiguously_and_reraises():
    """devices= plumbing of the *_batched entry points (no GPU: fake contexts)."""
    import threading

    from linalg_b200 import _native as nat

    seen, lock = [], threading.Lock()

    def fn(ctx, lo, hi):
        with lock:
            seen.append((ctx, lo, hi, threading.current_thread().name))

    nat.fan_out([3, 5, 6], 10, fn, _contexts=["c3", "c5", "c6"])
    assert sorted((c, lo, hi) for c, lo, hi, _ in seen) == [("c3", 0, 4), ("c5", 4, 7), ("c6", 7, 10)]
    assert len({name for *_, name in seen}) == 3            # one host thread per device
    seen.clear()
    nat.fan_out([0, 1, 2, 3], 2, fn, _contexts="abcd")      # more devices than units: empty slices are skipped
    assert sorted((lo, hi) for _, lo, hi, _ in seen) == [(0, 1), (1, 2)]

    def boom(ctx, lo, hi):
        if ctx == "b":
            raise ValueError("Input vectors are linearly dependent")

    with pytest.raises(ValueError, match="linearly dependent"):
        nat.fan_out([0, 1], 8, boom, _contexts="ab")
    with pytest.raises(ValueError):
        nat.fan_out([1, 1], 8, fn, _contexts="ab")
    with pytest.raises(ValueError):
        nat.fan_out([], 8, fn)


def test_native_environment_switches_are_the_documented_ones():
    """Kernel selection depends on the input shape: the native sources read only the switches of DESIGN.md §5 that select
    nothing or that the GPU tests use to reach a path well-conditioned input does not take."""
    import glob
    import re

    found = set()
    for path in glob.glob(os.path.join(ROOT, "linalg_b200", "csrc", "*.cu*")):
        with open(path) as fh:
            found |= set(re.findall(r"LINALG_B200_([A-Z_]+)", fh.read()))
    assert found == {"TRACE_BLOCKS", "NO_GRAPH", "TSQR_HOUSEHOLDER", "JACOBI_TWO_SIDED", "NCCL_LIB"}


def test_every_kernel_launch_goes_through_the_counted_helper():
    """launch / launch_cluster (ops.cuh) set a kernel's attributes once per device, launch it, check the launch and count
    it, so lq_kernel_launches counts exactly the kernels that ran.  Only the uncounted measurement utilities of api_core.cu
    launch directly; the launch count is otherwise written by the CUDA-graph replay alone; per-device state lives in the
    helper's bounds-checked, atomic DeviceLatch or in the context, never in a static table indexed by the device."""
    import glob
    import re

    src = {}
    for path in glob.glob(os.path.join(ROOT, "linalg_b200", "csrc", "*.cu*")):
        with open(path) as fh:
            src[os.path.basename(path)] = fh.read()

    def files_with(pattern):
        return {name for name, text in src.items() if re.search(pattern, text)}

    assert files_with(r"<<<|cudaLaunchKernelEx") == {"ops.cuh", "api_core.cu"}
    assert files_with(r"cudaFuncSetAttribute|DeviceLatch") == {"ops.cuh"}
    writes = {(name, m.group(0)) for name, text in src.items()
              for m in re.finditer(r"\w+(?:->|\.)launches\s*(?:\+\+|--|[-+]=|=(?!=))[^;]*", text)}
    assert writes == {
        ("ops.cuh", "c->launches++"),
        ("blocked_qr.cu", "c->launches += e->launches"),    # graph replay
        ("blocked_qr.cu", "e->launches = c->launches - l0"),  # graph capture
        ("blocked_qr.cu", "c->launches = l0"),              # capture failed: the plain path counts again
    }
    assert not files_with(r"static\s[^;(){}]*\[\s*64\s*\]")

"""ctypes binding of ``liblinalg_b200.so`` (the C ABI declared in ``include/linalg_b200.h``).

There is no CPU implementation behind this module: if the shared library is missing, or no
B200 is visible, the first call raises.  PyTorch is not imported.
"""
from __future__ import annotations

import ctypes as C
import os
import threading
import weakref

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_lib", "liblinalg_b200.so")

c_double_p = C.POINTER(C.c_double)
c_int32_p = C.POINTER(C.c_int32)
c_void_pp = C.POINTER(C.c_void_p)

# name -> (restype, argtypes); mirrors include/linalg_b200.h one to one
_CTX = C.c_void_p
_DP = C.c_void_p  # double* (host or device), passed as an address
SIGNATURES = {
    "lq_version": (C.c_char_p, []),
    "lq_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "lq_create": (C.c_int, [C.c_int, c_void_pp]),
    "lq_destroy": (C.c_int, [_CTX]),
    "lq_last_error": (C.c_char_p, [_CTX]),
    "lq_set_option": (C.c_int, [_CTX, C.c_char_p, C.c_int]),
    "lq_device_props": (C.c_int, [_CTX, C.POINTER(C.c_int64)]),
    "lq_malloc": (C.c_int, [_CTX, C.c_size_t, c_void_pp]),
    "lq_free": (C.c_int, [_CTX, C.c_void_p]),
    "lq_host_alloc": (C.c_int, [C.c_size_t, c_void_pp]),
    "lq_host_free": (C.c_int, [C.c_void_p]),
    "lq_memcpy_h2d": (C.c_int, [_CTX, C.c_void_p, C.c_void_p, C.c_size_t]),
    "lq_memcpy_d2h": (C.c_int, [_CTX, C.c_void_p, C.c_void_p, C.c_size_t]),
    "lq_memcpy_d2d": (C.c_int, [_CTX, C.c_void_p, C.c_void_p, C.c_size_t]),
    "lq_memset": (C.c_int, [_CTX, C.c_void_p, C.c_int, C.c_size_t]),
    "lq_sync": (C.c_int, [_CTX]),
    "lq_event_record": (C.c_int, [_CTX, C.c_int]),
    "lq_event_elapsed_ms": (C.c_int, [_CTX, C.c_int, C.c_int, C.POINTER(C.c_float)]),
    "lq_flush_l2": (C.c_int, [_CTX]),
    "lq_kernel_launches": (C.c_int64, [_CTX]),
    "lq_householder_qr_batched_dev": (C.c_int, [_CTX, _DP, C.c_int64, C.c_int, C.c_int, _DP, _DP, C.c_int]),
    "lq_householder_qr_batched": (C.c_int, [_CTX, _DP, C.c_int64, C.c_int, C.c_int, _DP, _DP]),
    "lq_householder_qr_dev": (C.c_int, [_CTX, _DP, C.c_int, C.c_int, _DP, _DP]),
    "lq_householder_qr": (C.c_int, [_CTX, _DP, C.c_int, C.c_int, _DP, _DP]),
    "lq_mgs_qr_batched_dev": (C.c_int, [_CTX, _DP, C.c_int64, C.c_int, C.c_int, C.c_int, _DP, _DP, C.c_void_p]),
    "lq_mgs_qr_batched": (C.c_int, [_CTX, _DP, C.c_int64, C.c_int, C.c_int, C.c_int, _DP, _DP, C.c_void_p]),
    "lq_mgs_qr_dev": (C.c_int, [_CTX, _DP, C.c_int, C.c_int, C.c_int, _DP, _DP, C.c_void_p]),
    "lq_mgs_qr": (C.c_int, [_CTX, _DP, C.c_int, C.c_int, C.c_int, _DP, _DP, C.c_void_p]),
    "lq_lstsq_householder_batched_dev": (C.c_int, [_CTX, _DP, _DP, C.c_int64, C.c_int, C.c_int, C.c_int, _DP]),
    "lq_lstsq_householder_batched": (C.c_int, [_CTX, _DP, _DP, C.c_int64, C.c_int, C.c_int, C.c_int, _DP]),
    "lq_lstsq_householder_batched_info": (C.c_int, [_CTX, _DP, _DP, C.c_int64, C.c_int, C.c_int, C.c_int, _DP, _DP]),
    "lq_lstsq_householder_batched_info_dev": (C.c_int, [_CTX, _DP, _DP, C.c_int64, C.c_int, C.c_int, C.c_int, _DP, _DP]),
    "lq_lstsq_mgs_batched_dev": (C.c_int, [_CTX, _DP, _DP, C.c_int64, C.c_int, C.c_int, C.c_int, _DP, C.c_void_p]),
    "lq_lstsq_mgs_batched": (C.c_int, [_CTX, _DP, _DP, C.c_int64, C.c_int, C.c_int, C.c_int, _DP, C.c_void_p]),
    "lq_svd_gram_dev": (C.c_int, [_CTX, _DP, C.c_int64, C.c_int, C.c_double, _DP, _DP, _DP, C.POINTER(C.c_int)]),
    "lq_svd_gram": (C.c_int, [_CTX, _DP, C.c_int64, C.c_int, C.c_double, _DP, _DP, _DP, C.POINTER(C.c_int)]),
    "lq_svd_gram_batched_dev": (C.c_int, [_CTX, _DP, C.c_int64, C.c_int, C.c_int, C.c_double, _DP, _DP, _DP, C.c_void_p]),
    "lq_svd_gram_batched": (C.c_int, [_CTX, _DP, C.c_int64, C.c_int, C.c_int, C.c_double, _DP, _DP, _DP, C.c_void_p]),
    "lq_svd_complete": (C.c_int, [_CTX, _DP, C.c_int64, C.c_int, C.c_int, _DP]),
    "lq_svd_complete_seeded": (C.c_int, [_CTX, _DP, C.c_int64, C.c_int, C.c_int, C.c_uint64]),
    "lq_random_normal_dev": (C.c_int, [_CTX, _DP, C.c_int64, C.c_uint64]),
    "lq_gram_dev": (C.c_int, [_CTX, _DP, C.c_int64, C.c_int, _DP]),
    "lq_eigh_dev": (C.c_int, [_CTX, _DP, C.c_int, _DP, _DP]),
    "lq_gemm_dev": (C.c_int, [_CTX, C.c_int, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_double, _DP, C.c_int, _DP,
                              C.c_int, C.c_double, _DP, C.c_int]),
    "lq_tsqr_dev": (C.c_int, [_CTX, _DP, C.c_int64, C.c_int, _DP, _DP]),
    "lq_tsqr": (C.c_int, [_CTX, _DP, C.c_int64, C.c_int, _DP, _DP]),
    "lq_lstsq_tsqr_dev": (C.c_int, [_CTX, _DP, C.c_int64, C.c_int, _DP, C.c_int, _DP, C.c_void_p]),
    "lq_lstsq_tsqr": (C.c_int, [_CTX, _DP, C.c_int64, C.c_int, _DP, C.c_int, _DP, C.c_void_p]),
    "lq_comm_unique_id": (C.c_int, [C.c_void_p]),
    "lq_comm_init": (C.c_int, [_CTX, C.c_int, C.c_int, C.c_void_p]),
    "lq_comm_destroy": (C.c_int, [_CTX]),
    "lq_comm_allreduce_sum": (C.c_int, [_CTX, _DP, C.c_int64]),
    "lq_comm_allgather": (C.c_int, [_CTX, _DP, _DP, C.c_int64]),
    "lq_tsqr_sharded_dev": (C.c_int, [_CTX, _DP, C.c_int64, C.c_int, _DP, _DP]),
    "lq_svd_gram_sharded_dev": (C.c_int, [_CTX, _DP, C.c_int64, C.c_int, C.c_double, _DP, _DP, _DP,
                                          C.POINTER(C.c_int)]),
    "lq_lstsq_tsqr_sharded_dev": (C.c_int, [_CTX, _DP, C.c_int64, C.c_int, _DP, C.c_int, _DP, C.c_void_p]),
    "lq_probe": (C.c_int, [_CTX, C.c_int, C.POINTER(C.c_double)]),
    "lq_debug_panel_trace": (C.c_int, [_CTX, _DP, C.c_int, _DP, C.c_int, _DP, C.c_int, C.c_int, C.c_void_p]),
    "lq_debug_panel": (C.c_int, [_CTX, _DP, C.c_int, _DP, C.c_int, _DP, C.c_int, C.c_int, C.c_int, C.c_int]),
}

_lib = None
_lib_lock = threading.Lock()


class NativeLibraryMissing(RuntimeError):
    pass


def load_library():
    """dlopen the in-tree shared library and attach the signatures (no GPU needed for this)."""
    global _lib
    with _lib_lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise NativeLibraryMissing(
                f"{LIB_PATH} not found: build it with `python -m linalg_b200.build` "
                "(linalg_b200 has no CPU fallback)"
            )
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the ABI and the header drift apart
            fn.restype = res
            fn.argtypes = args
        _lib = lib
        return lib


def _err_text(lib, ctx) -> str:
    msg = lib.lq_last_error(ctx)
    return msg.decode("utf-8", "replace") if msg else ""


def check(lib, ctx, rc: int, what: str = ""):
    """Map a C-ABI status to the reference's exception classes."""
    if rc == 0:
        return
    text = _err_text(lib, ctx)
    if rc < 0:
        if rc == -3:
            raise NotImplementedError(f"{what}: {text} (status {rc})")
        raise ValueError(f"{what}: {text} (status {rc})")
    raise RuntimeError(f"{what}: {text} (status {rc})")


class DeviceBuffer:
    """A cudaMalloc'ed region owned by a Context."""

    def __init__(self, ctx: "Context", nbytes: int):
        self.ctx = ctx
        self.nbytes = int(nbytes)
        p = C.c_void_p()
        check(ctx.lib, ctx.handle, ctx.lib.lq_malloc(ctx.handle, self.nbytes, C.byref(p)), "lq_malloc")
        self.ptr = p.value

    def free(self):
        if self.ptr:
            self.ctx.lib.lq_free(self.ctx.handle, self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Context:
    """One device + one stream + scratch (+ optional NCCL communicator)."""

    def __init__(self, device: int = 0):
        self.lib = load_library()
        h = C.c_void_p()
        rc = self.lib.lq_create(int(device), C.byref(h))
        if rc != 0:
            raise RuntimeError(
                f"lq_create(device={device}) failed: {_err_text(self.lib, None)} (status {rc}); "
                "linalg_b200 needs a B200 (sm_100a) and has no CPU fallback"
            )
        self.handle = h
        self.device = int(device)

    # -- plumbing ---------------------------------------------------------------------
    def close(self):
        if getattr(self, "handle", None):
            self.lib.lq_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def call(self, name: str, *args):
        rc = getattr(self.lib, name)(self.handle, *args)
        check(self.lib, self.handle, rc, name)

    def set_option(self, name: str, value: bool):
        """Diagnostic kernel-selection switch (``TSQR_HOUSEHOLDER`` or ``JACOBI_TWO_SIDED``); any other name raises ValueError."""
        self.call("lq_set_option", name.encode(), int(bool(value)))

    def props(self):
        arr = (C.c_int64 * 8)()
        self.call("lq_device_props", arr)
        keys = ["sm_count", "cc_major", "cc_minor", "max_smem", "sm_clock_khz", "mem_mib", "l2_bytes", "max_cluster"]
        return dict(zip(keys, [int(v) for v in arr]))

    def alloc(self, nbytes: int) -> DeviceBuffer:
        return DeviceBuffer(self, nbytes)

    def upload(self, arr: np.ndarray, buf: DeviceBuffer | None = None) -> DeviceBuffer:
        arr = np.ascontiguousarray(arr)
        if buf is None:
            buf = self.alloc(arr.nbytes)
        self.call("lq_memcpy_h2d", buf.ptr, arr.ctypes.data, arr.nbytes)
        self.sync()
        return buf

    def download(self, buf: DeviceBuffer, shape, dtype=np.float64, out: np.ndarray | None = None) -> np.ndarray:
        if out is None:
            out = np.empty(shape, dtype=dtype)
        self.call("lq_memcpy_d2h", out.ctypes.data, buf.ptr, out.nbytes)
        self.sync()
        return out

    def sync(self):
        self.call("lq_sync")

    def record(self, slot: int):
        self.call("lq_event_record", int(slot))

    def elapsed_ms(self, a: int, b: int) -> float:
        ms = C.c_float()
        self.call("lq_event_elapsed_ms", int(a), int(b), C.byref(ms))
        return float(ms.value)

    def flush_l2(self):
        self.call("lq_flush_l2")

    def launches(self) -> int:
        return int(self.lib.lq_kernel_launches(self.handle))

    def probe(self, kind: int) -> float:
        v = C.c_double()
        self.call("lq_probe", int(kind), C.byref(v))
        return float(v.value)


_default_ctx = None
_default_lock = threading.Lock()


def default_context() -> Context:
    """Process-wide context on device ``$LINALG_B200_DEVICE`` (or ``$LOCAL_RANK``, else 0)."""
    global _default_ctx
    with _default_lock:
        if _default_ctx is None:
            dev = int(os.environ.get("LINALG_B200_DEVICE", os.environ.get("LOCAL_RANK", "0")))
            _default_ctx = Context(dev)
        return _default_ctx


_device_ctxs: dict = {}


def device_context(device: int) -> Context:
    """Process-wide context of one device (created on first use); the default context is reused for its device."""
    device = int(device)
    with _default_lock:
        if _default_ctx is not None and _default_ctx.device == device:
            return _default_ctx
        ctx = _device_ctxs.get(device)
        if ctx is None:
            ctx = _device_ctxs[device] = Context(device)
        return ctx


def device_count() -> int:
    n = C.c_int(0)
    lib = load_library()
    check(lib, None, lib.lq_device_count(C.byref(n)), "lq_device_count")
    return int(n.value)


def fan_out(devices, total: int, fn, _contexts=None):
    """Run ``fn(ctx, lo, hi)`` for a contiguous split of ``range(total)`` over ``devices`` -- one host thread and one
    context per device, no communication (SURVEY.md section 8e: batched problems shard by batch index).  ctypes drops
    the GIL inside the C call, so the per-device host-pointer pipelines (H2D, kernels, D2H) run concurrently.  The
    first exception of any device is re-raised after every thread has finished."""
    from .utils import shard_bounds

    devices = [int(d) for d in devices]
    if not devices:
        raise ValueError("devices must name at least one GPU")
    if len(set(devices)) != len(devices):
        raise ValueError(f"devices must be distinct, got {devices}")
    ctxs = [device_context(d) for d in devices] if _contexts is None else list(_contexts)
    parts = [shard_bounds(total, len(devices), r) for r in range(len(devices))]
    errors = [None] * len(devices)

    def work(r):
        lo, hi = parts[r]
        if hi > lo:
            try:
                fn(ctxs[r], lo, hi)
            except BaseException as exc:  # noqa: BLE001 -- re-raised in the caller's thread
                errors[r] = exc

    threads = [threading.Thread(target=work, args=(r,), name=f"linalg_b200-dev{devices[r]}") for r in range(1, len(devices))]
    for t in threads:
        t.start()
    work(0)
    for t in threads:
        t.join()
    for exc in errors:
        if exc is not None:
            raise exc


def pinned_empty(shape, dtype=np.float64) -> np.ndarray:
    """NumPy array over page-locked host memory (fast, truly asynchronous H2D/D2H)."""
    lib = load_library()
    dtype = np.dtype(dtype)
    n = int(np.prod(shape)) * dtype.itemsize
    p = C.c_void_p()
    rc = lib.lq_host_alloc(max(n, 16), C.byref(p))
    if rc != 0:
        raise MemoryError(f"lq_host_alloc({n}) failed: {_err_text(lib, None)}")
    buf = (C.c_char * max(n, 16)).from_address(p.value)
    # the ctypes block is the root owner of every view; free the pinned memory when it dies
    weakref.finalize(buf, lib.lq_host_free, p.value)
    return np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

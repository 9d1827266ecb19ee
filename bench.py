#!/usr/bin/env python3
"""Benchmark of the dense-factorisation hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--no-extras] [--dump-outputs DIR]

Headline workload (BASELINE.json configs[1], the one the metric is quoted on): batched Householder
QR of 2^20 independent 32 x 32 float64 matrices per GPU; one "step" = one pass over that batch.
N > 1 (launched by torchrun, one rank per GPU): the batch index is sharded, every rank factors its
own 2^20 matrices with no data-path collective ("scaling": "weak"); the timed region is bracketed
by a barrier + stream synchronisation and the reported time is the max over ranks.

value   = matrices/s with the inputs already resident in HBM (CUDA events on the library's stream)
e2e     = the same metric through the host-pointer C-ABI call lq_householder_qr_batched (pinned
          NumPy buffers, H2D of A and D2H of Q and R inside the timed region, every step)
roofline, cpu_baseline, clocks, gpu_launches: see DESIGN.md "Measurement".
extras  = the other BASELINE configs (MGS, least squares, blocked 8192^2, tall-skinny TSQR / SVD)
          measured the same way, each with its own roofline fraction.

--dump-outputs DIR writes Q and R of the last timed step for a fixed, seeded sample of DUMP_MATRICES matrices
(rank 0's batch) as DIR/Q.npy and DIR/R.npy, float64.  The inputs depend on the arguments only, so two builds
of the project can be compared output for output.

--impl reference times the reference's CPU algorithm (the NumPy oracle port -- the reference is
pure Python and cannot travel to the GPU box) on all host cores, on a bounded sample of the same
workload; under torchrun only rank 0 runs it.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N32 = 32
BYTES_PER_MATRIX = 8 * 3 * N32 * N32            # read A, write Q, write dense R  (BASELINE.md section 4)
FLOPS_HH32 = 87381                               # F_QR(32, 32)
FLOPS_MGS32 = 65536
PER_GPU_BATCH = 1 << 20
UNIQUE = 1 << 16                                 # distinct random matrices, tiled to the full batch
DUMP_MATRICES = 2048                             # --dump-outputs sample: 2 x 2048 x 8 KiB = 32 MiB


def _json_default(o):
    """NumPy scalars (np.bool_, np.float64, np.int64) that slipped into the line."""
    if hasattr(o, "item"):
        return o.item()
    raise TypeError(f"not JSON serialisable: {type(o).__name__}")


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            d = json.load(open(path))
            return {"hbm_gbs": float(d["hbm_gbs"]), "source": "measured (MEASURED_PEAKS.json)"}
        except Exception:
            pass
    return {"hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md)"}


def profile_traffic(kernel_key):
    """DRAM bytes per launch of the dominant kernel from the committed ncu capture, or None."""
    path = os.path.join(ROOT, "profiles", "roofline_traffic.json")
    try:
        return json.load(open(path)).get(kernel_key)
    except Exception:
        return None


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.device}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "25"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def mark(self):
        return time.time()

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self, t0, t1):
        sm, smmax, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.rows:
            if ts < t0 or ts > t1 + 0.15:
                continue
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                smmax = max(smmax, float(parts[1]))
            except ValueError:
                continue
            for nme, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(nme)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": smmax, "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------- CPU baseline (oracle port)
def _cpu_worker(args):
    kind, seed, count = args
    os.environ["OPENBLAS_NUM_THREADS"] = "1"
    from oracle import linalg_oracle as orc

    rng = np.random.default_rng(seed)
    if kind == "hh32":
        A = rng.standard_normal((count, N32, N32))
        t = time.perf_counter()
        for i in range(count):
            orc.householder_qr(A[i])
        return time.perf_counter() - t
    raise ValueError(kind)


def cpu_baseline_hh32(per_worker=16384, workers=None, steps=1, warmup=0):
    """The reference's algorithm (NumPy oracle port, linalg/qr.py:52-100) over all host cores:
    one process per core, BLAS pinned to 1 thread each (BASELINE.md section 5).  One "step" factors
    ``per_worker * workers`` matrices; returns the mean throughput of the timed steps."""
    import concurrent.futures as cf
    import multiprocessing as mp

    workers = workers or (os.cpu_count() or 1)
    workers = min(workers, 64)
    os.environ["OPENBLAS_NUM_THREADS"] = "1"
    os.environ["OMP_NUM_THREADS"] = "1"
    os.environ["MKL_NUM_THREADS"] = "1"
    ctxm = mp.get_context("spawn")
    walls, slowest = [], 0.0
    with cf.ProcessPoolExecutor(max_workers=workers, mp_context=ctxm) as ex:
        list(ex.map(_cpu_worker, [("hh32", 1, 8)] * workers))  # import + warm-up, untimed
        for it in range(warmup + steps):
            t1 = time.perf_counter()
            times = list(ex.map(_cpu_worker, [("hh32", 2 + w + 100 * it, per_worker) for w in range(workers)]))
            if it >= warmup:
                walls.append(time.perf_counter() - t1)
                slowest = max(slowest, max(times))
    total = per_worker * workers
    wall = statistics.mean(walls)
    return {
        "value": total / wall,
        "unit": "matrices/s",
        "cores": workers,
        "kind": "port",
        "sample": f"{total} of the 2^20 32x32 matrices per step ({per_worker} per process x {workers} processes, "
                  f"OPENBLAS_NUM_THREADS=1), NumPy oracle of linalg/qr.py:52-100; {len(walls)} step(s), "
                  f"mean wall {wall:.2f} s, slowest worker {slowest:.2f} s",
        "host_cpu_count": os.cpu_count(),
    }


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    per_worker = 1024   # x cores matrices per step; the default 20 + 5 steps then take ~15-20 s
    base = cpu_baseline_hh32(per_worker=per_worker, steps=args.steps, warmup=args.warmup)
    value = base["value"]
    line = {
        "impl": "reference",
        "metric": "batched Householder QR throughput, 32x32 float64",
        "value": value,
        "unit": "matrices/s",
        "n_gpus": args.gpus,
        "steps": args.steps,
        "warmup": args.warmup,
        "ms_per_step": 1e3 * per_worker * base["cores"] / value,
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": "f64",
        "data": "synthetic (default_rng standard_normal)",
        "config": {"workload": "cfg2: batched householder_qr of 2^20 independent 32x32 float64 matrices per GPU "
                               "(CPU arm: bounded sample per step)",
                   "sample_per_step": per_worker * base["cores"]},
        "cpu_baseline": base,
        "e2e": {"value": value, "unit": "matrices/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line, default=_json_default), flush=True)
    return 0


# ----------------------------------------------------------------------------- device helpers
def timed(ctx, fn, steps, warmup, flush=False):
    """Run fn() warmup+steps times on the context stream; returns (list of per-step ms, total ms)."""
    for _ in range(warmup):
        fn()
    ctx.sync()
    per = []
    for i in range(steps):
        if flush:
            ctx.flush_l2()
        ctx.record(0)
        fn()
        ctx.record(1)
        per.append(ctx.elapsed_ms(0, 1))
    return per


def host_memory_budget_bytes():
    """Bytes of host RAM this process may safely pin: min(MemAvailable, cgroup limit - usage) / 2."""
    avail = None
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable:"):
                avail = int(line.split()[1]) * 1024
    except OSError:
        pass
    for lim_path, use_path in (("/sys/fs/cgroup/memory.max", "/sys/fs/cgroup/memory.current"),
                               ("/sys/fs/cgroup/memory/memory.limit_in_bytes", "/sys/fs/cgroup/memory/memory.usage_in_bytes")):
        try:
            lim = open(lim_path).read().strip()
            if lim != "max":
                room = int(lim) - int(open(use_path).read().strip())
                avail = room if avail is None else min(avail, room)
        except (OSError, ValueError):
            pass
    return (avail if avail is not None else 16 << 30) // 2


def tile_to_device(ctx, block: np.ndarray, reps: int):
    per = block.nbytes
    buf = ctx.alloc(per * reps)
    ctx.call("lq_memcpy_h2d", buf.ptr, block.ctypes.data, per)
    for r in range(1, reps):
        ctx.call("lq_memcpy_d2d", buf.ptr + r * per, buf.ptr, per)
    ctx.sync()
    return buf


def dump_outputs(ctx, out_dir, dQ, dR, batch):
    """Q and R of DUMP_MATRICES matrices of the batch, drawn with a fixed seed across all of it (the tiled replicas
    included), -> out_dir/Q.npy, out_dir/R.npy as (count, 32, 32) float64 in ascending batch order."""
    idx = np.sort(np.random.default_rng(0).choice(batch, size=min(DUMP_MATRICES, batch), replace=False))
    per = 8 * N32 * N32
    os.makedirs(out_dir, exist_ok=True)
    for name, buf in (("Q", dQ), ("R", dR)):
        out = np.empty((len(idx), N32, N32))
        for k, i in enumerate(idx):
            ctx.call("lq_memcpy_d2h", out[k].ctypes.data, buf.ptr + int(i) * per, per)
        ctx.sync()
        np.save(os.path.join(out_dir, f"{name}.npy"), out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-extras", action="store_true", help="skip the secondary configs (cfg1/3/4/5)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg")
    ap.add_argument("--e2e-steps", type=int, default=0, help="end-to-end steps (default min(steps, 5))")
    ap.add_argument("--batch", type=int, default=PER_GPU_BATCH, help="matrices per GPU")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write Q and R of the last timed step (a fixed sample of the batch) as DIR/Q.npy, DIR/R.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    if args.impl == "reference":
        return run_reference_arm(args)

    # libraries underneath (NCCL prints its version banner) may write to stdout: keep fd 1 clean for the JSON line
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    import linalg_b200 as lb
    from linalg_b200 import dist as d

    info = d.init_control_plane("gloo")
    if info.world != args.gpus and info.world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={info.world}")
    peaks = measured_peaks()

    # CPU baseline first (rank 0, N = 1 only): process pool, before the CUDA context exists
    cpu = None
    if info.rank == 0 and info.world == 1 and not args.no_cpu:
        cpu = cpu_baseline_hh32()

    ctx = lb.Context(info.local_rank)
    props = ctx.props()
    batch = args.batch
    uniq = min(UNIQUE, batch)
    reps = batch // uniq
    batch = uniq * reps
    rng = np.random.default_rng(2 + 1000 * info.rank)
    block = rng.standard_normal((uniq, N32, N32))
    dA = tile_to_device(ctx, block, reps)
    dQ, dR = ctx.alloc(block.nbytes * reps), ctx.alloc(block.nbytes * reps)

    def step_hh():
        ctx.call("lq_householder_qr_batched_dev", dA.ptr, batch, N32, N32, dQ.ptr, dR.ptr, 0)

    sampler = ClockSampler(info.local_rank)
    sampler.start()
    time.sleep(0.3)          # let the sampler produce its first rows
    c0 = sampler.mark()      # clocks are sampled from the warm-up through the timed region (it lasts only ~0.1-0.2 s)
    for _ in range(args.warmup):
        step_hh()
    ctx.sync()
    d.barrier()
    l0 = ctx.launches()
    ctx.record(2)
    for _ in range(args.steps):
        step_hh()
    ctx.record(3)
    ctx.sync()
    total_ms = ctx.elapsed_ms(2, 3)
    c1 = sampler.mark()
    launches = ctx.launches() - l0
    d.barrier()
    total_ms_max = d.max_over_ranks(total_ms)
    ms_per_step = total_ms_max / args.steps
    value = info.world * batch / (ms_per_step * 1e-3)
    kernel_ms = total_ms / args.steps            # one launch per step: the bracket IS the kernel time
    achieved = batch * BYTES_PER_MATRIX / (kernel_ms * 1e-3) / 1e9
    clocks = sampler.summary(c0, c1)

    # sanity: the timed kernel really produced a factorisation (first matrices of the batch)
    nchk = 64
    Qh, Rh = np.empty((nchk, N32, N32)), np.empty((nchk, N32, N32))
    ctx.call("lq_memcpy_d2h", Qh.ctypes.data, dQ.ptr, Qh.nbytes)
    ctx.call("lq_memcpy_d2h", Rh.ctypes.data, dR.ptr, Rh.nbytes)
    ctx.sync()
    resid = float(np.max(np.linalg.norm(block[:nchk] - Qh @ Rh, axis=(1, 2)) / np.linalg.norm(block[:nchk], axis=(1, 2))))
    if not resid < 1e-12:
        raise SystemExit(f"bench: factorisation check failed (residual {resid})")
    if args.dump_outputs and info.rank == 0:
        dump_outputs(ctx, args.dump_outputs, dQ, dR, batch)   # before the MGS leg below overwrites dQ, dR

    extras = {"hh32_residual_check": resid}

    # ---- MGS on the same batch (cfg2, second half)
    dI = ctx.alloc(4 * batch)
    ms = timed(ctx, lambda: ctx.call("lq_mgs_qr_batched_dev", dA.ptr, batch, N32, N32, 0, dQ.ptr, dR.ptr, dI.ptr),
               max(3, args.steps // 2), 3)
    mgs_ms = d.max_over_ranks(statistics.mean(ms))
    extras["cfg2_mgs32"] = {
        "matrices_per_s": info.world * batch / (mgs_ms * 1e-3), "ms": mgs_ms,
        "hbm_gbs_per_gpu": batch * BYTES_PER_MATRIX / (mgs_ms * 1e-3) / 1e9,
        "hbm_frac": batch * BYTES_PER_MATRIX / (mgs_ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
        "gflops": info.world * batch * FLOPS_MGS32 / (mgs_ms * 1e-3) / 1e9,
    }
    dI.free()

    # ---- cfg2 strong scaling: 2^20 matrices IN TOTAL, batch-sharded over the ranks (no collective); every step is
    # bracketed by a barrier so launch / barrier overhead shows (1.2 ms kernels at N = 8)
    sb = PER_GPU_BATCH // info.world
    if sb <= batch:
        per = []
        for i in range(3 + 10):
            ctx.sync()
            d.barrier()
            ctx.record(0)
            ctx.call("lq_householder_qr_batched_dev", dA.ptr, sb, N32, N32, dQ.ptr, dR.ptr, 0)
            ctx.record(1)
            ctx.sync()
            if i >= 3:
                per.append(d.max_over_ranks(ctx.elapsed_ms(0, 1)))
        sms = statistics.mean(per)
        extras["cfg2_strong_1M_total"] = {"matrices_total": sb * info.world, "matrices_per_gpu": sb, "ms": sms,
                                          "matrices_per_s": sb * info.world / (sms * 1e-3), "scaling": "strong",
                                          "hbm_frac_per_gpu": sb * BYTES_PER_MATRIX / (sms * 1e-3) / 1e9 / peaks["hbm_gbs"]}

    # ---- end to end: pinned host buffers through the host-pointer C-ABI call
    e2e_steps = args.e2e_steps or min(args.steps, 5)
    budget = host_memory_budget_bytes() // max(1, info.world)
    e2e_reps = max(1, min(reps, budget // (3 * block.nbytes)))   # full batch unless host RAM is short
    e2e_batch = uniq * e2e_reps
    hA = lb.pinned_empty((e2e_batch, N32, N32))
    hQ = lb.pinned_empty((e2e_batch, N32, N32))
    hR = lb.pinned_empty((e2e_batch, N32, N32))
    for r in range(e2e_reps):
        hA[r * uniq:(r + 1) * uniq] = block

    def step_e2e():
        ctx.call("lq_householder_qr_batched", hA.ctypes.data, e2e_batch, N32, N32, hQ.ctypes.data, hR.ctypes.data)

    step_e2e()  # warm-up (allocates the staging lanes)
    d.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        step_e2e()
    e2e_s = d.max_over_ranks(time.perf_counter() - t0)
    e2e_value = info.world * e2e_batch * e2e_steps / e2e_s
    resid2 = float(np.max(np.linalg.norm(hA[-4:] - hQ[-4:] @ hR[-4:], axis=(1, 2)) / np.linalg.norm(hA[-4:], axis=(1, 2))))
    if not resid2 < 1e-12:
        raise SystemExit(f"bench: e2e factorisation check failed (residual {resid2})")
    e2e = {"value": e2e_value, "unit": "matrices/s", "h2d_bytes_per_step": int(hA.nbytes),
           "d2h_bytes_per_step": int(hQ.nbytes + hR.nbytes), "steps": e2e_steps, "batch_per_gpu": e2e_batch,
           "pcie_gbs": (hA.nbytes + hQ.nbytes + hR.nbytes) * e2e_steps / e2e_s / 1e9,
           "api": "lq_householder_qr_batched (host pointers, pinned NumPy buffers)"}
    # the host side's ceiling for this call: the same bytes (A up, Q and R down) as plain cudaMemcpyAsync copies from / to the
    # same pinned buffers, H2D and D2H on two streams, all ranks at once -- no kernels.  e2e / ceiling says how much of the
    # copy roof the pipeline reaches; ceiling(N) / ceiling(1) says what the box's host memory / PCIe fabric gives N GPUs.
    try:
        nb = min(e2e_batch, batch) * N32 * N32 * 8
        ctx2 = lb.Context(ctx.device)
        best = None
        for _ in range(3):
            ctx.sync(); ctx2.sync()
            d.barrier()
            t0 = time.perf_counter()
            ctx.call("lq_memcpy_h2d", dA.ptr, hA.ctypes.data, nb)
            ctx2.call("lq_memcpy_d2h", hQ.ctypes.data, dQ.ptr, nb)
            ctx2.call("lq_memcpy_d2h", hR.ctypes.data, dR.ptr, nb)
            ctx.sync(); ctx2.sync()
            dt = d.max_over_ranks(time.perf_counter() - t0)
            best = dt if best is None else min(best, dt)
        ceil_gbs = info.world * 3 * nb / best / 1e9
        e2e["copy_ceiling"] = {"all_ranks_gbs": ceil_gbs, "per_gpu_gbs": ceil_gbs / info.world,
                               "e2e_frac_of_ceiling": e2e["pcie_gbs"] * info.world / ceil_gbs,
                               "how": "cudaMemcpyAsync of A (H2D) and Q, R (D2H) on two streams from the same pinned buffers, all ranks concurrently, best of 3"}
        ctx2.close()
    except Exception as exc:  # diagnostics only
        e2e["copy_ceiling"] = {"error": repr(exc)}
    # the in-process multi-GPU form of the same call (SURVEY.md section 5: `devices=`): rank 0 alone fans a 2^18-matrix batch
    # over every GPU of the launch from ONE process (one host thread + context per GPU, no communication) while the other
    # ranks wait; the result is compared with the single-GPU call bit for bit
    if info.world > 1 and not args.no_extras:
        try:
            from linalg_b200 import _native as _nat

            ndev = min(info.world, _nat.device_count())
            d.barrier()
            if info.rank == 0 and ndev > 1:
                nb = min(1 << 18, e2e_batch)
                devs = [ctx.device] + [k for k in range(ndev) if k != ctx.device]
                Q1, R1 = lb.householder_qr_batched(hA[:nb], out=(hQ[:nb], hR[:nb]), ctx=ctx)
                Qd, Rd = lb.pinned_empty((nb, N32, N32)), lb.pinned_empty((nb, N32, N32))
                lb.householder_qr_batched(hA[:nb], out=(Qd, Rd), devices=devs)          # warm-up: contexts, staging lanes
                t0 = time.perf_counter()
                for _ in range(3):
                    lb.householder_qr_batched(hA[:nb], out=(Qd, Rd), devices=devs)
                dt = (time.perf_counter() - t0) / 3
                t0 = time.perf_counter()
                for _ in range(3):
                    lb.householder_qr_batched(hA[:nb], out=(hQ[:nb], hR[:nb]), ctx=ctx)
                dt1 = (time.perf_counter() - t0) / 3
                same = bool(np.array_equal(Qd, Q1) and np.array_equal(Rd, R1))
                _require(same, "devices= result bitwise equal to the one-GPU call", same)
                e2e["devices_kwarg"] = {"devices": devs, "batch": nb, "matrices_per_s": nb / dt, "one_gpu_matrices_per_s": nb / dt1,
                                        "bitwise_equal_to_one_gpu": same,
                                        "api": "householder_qr_batched(A, devices=[...]) from ONE process, the other ranks idle"}
                del Qd, Rd
            d.barrier()
        except ParityError:
            raise
        except Exception as exc:  # diagnostics only
            e2e["devices_kwarg"] = {"error": repr(exc)}
            d.barrier()
    del hA, hQ, hR
    dA.free(); dQ.free(); dR.free()

    if not args.no_extras:
        try:
            extras.update(run_extras(ctx, d, info, peaks))
        except ParityError:
            raise                  # a timed configuration with a wrong result fails the run
        except Exception as exc:  # anything else in the extras must never lose the headline line
            extras["extras_error"] = repr(exc)

    sampler.stop()
    if info.rank == 0:
        fp64 = extras.get("fp64_peaks", {})
        line = {
            "metric": "batched Householder QR throughput, 32x32 float64",
            "value": value,
            "unit": "matrices/s",
            "n_gpus": info.world,
            "steps": args.steps,
            "warmup": args.warmup,
            "ms_per_step": ms_per_step,
            "higher_is_better": True,
            "scaling": "weak",
            "vs_baseline": None,
            "dtype": "f64",
            "data": f"synthetic: default_rng(2+1000*rank).standard_normal, {uniq} distinct matrices tiled x{reps}",
            "config": {
                "workload": "cfg2: batched householder_qr of 2^20 independent 32x32 float64 matrices per GPU",
                "per_gpu_batch": batch, "global_batch": batch * info.world, "parallelism": f"batch-sharded x{info.world}, no collective",
                "l2": "inputs 8.6 GB per GPU >> 126 MB L2 (no flush needed)",
                "gflops": value * FLOPS_HH32 / 1e9,
            },
            "roofline": {
                "bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": achieved / peaks["hbm_gbs"], "traffic": profile_traffic("hh_qr32_c8_kernel"),
                "peak_source": peaks["source"], "kernel": "hh_qr32_c8_kernel<8,1,3,true>", "kernel_ms": kernel_ms,
                "algorithmic_bytes_per_launch": batch * BYTES_PER_MATRIX,
                "frac_of_nominal_8TBs": achieved / 8000.0,
                "fp64_frac": (batch * FLOPS_HH32 / (kernel_ms * 1e-3) / 1e12 / fp64["dfma_tflops"]) if fp64.get("dfma_tflops") else None,
            },
            "cpu_baseline": cpu,
            "e2e": e2e,
            "gpu_launches": int(launches),
            "clocks": clocks,
            "device": {"sm_count": props["sm_count"], "cc": f"{props['cc_major']}.{props['cc_minor']}", "mem_mib": props["mem_mib"]},
            "extras": extras,
        }
        os.write(json_fd, (json.dumps(line, default=_json_default) + "\n").encode())
    d.barrier()
    ctx.close()
    d.shutdown_control_plane()
    return 0


# ----------------------------------------------------------------------------- parity of the timed outputs
class ParityError(RuntimeError):
    """A timed configuration produced a result outside the north-star tolerances: the run must fail."""


def _require(cond, what, value):
    if not cond:
        raise ParityError(f"bench parity check failed: {what} = {value}")


def _gram_all(ctx, info, dX, m, n):
    """G = X^T X over ALL row shards: device Gram (+ one ncclAllReduce of n*n doubles), downloaded."""
    dG = ctx.alloc(8 * n * n)
    ctx.call("lq_gram_dev", dX.ptr, m, n, dG.ptr)
    if info.world > 1:
        ctx.call("lq_comm_allreduce_sum", dG.ptr, n * n)
    G = ctx.download(dG, (n, n))
    dG.free()
    return G


def _row_sample(ctx, dX, m, n, rows=4096):
    """First / middle / last `rows` rows of a device (m, n) array -> host."""
    rows = min(rows, m)
    starts = sorted({0, max(0, m // 2 - rows // 2), m - rows})
    out = np.empty((len(starts) * rows, n))
    for k, st in enumerate(starts):
        ctx.call("lq_memcpy_d2h", out[k * rows:].ctypes.data, dX.ptr + 8 * st * n, 8 * rows * n)
    ctx.sync()
    idx = np.concatenate([np.arange(st, st + rows) for st in starts])
    return idx, out


def check_cfg5(ctx, d, info, A, dA, dQ, dR, dU, ds, dVt, m, n):
    """Checked results behind the tall-skinny timings (north star: ||Q^T Q - I|| <= 1e-12, ||A - QR|| / ||A|| <= 1e-12,
    singular values to 1e-10 relative), valid for any number of row shards:
      orthogonality over ALL rows     Gram of Q / U on the device, all-reduced             (linalg/qr.py:39-42 convention)
      residual                        per rank on 3 x 4096 rows of its shard, and over all rows through
                                      A^T A = R^T R  /  A^T A = V diag(s^2) V^T           (linalg/svd.py:42-64)
      replication                     R, s, Vt bitwise identical on every rank
      s(svd route) vs s(R)            np.linalg.svd of the 128 x 128 TSQR factor (host)"""
    import hashlib

    eye = np.eye(n)
    out = {}
    # ---- TSQR
    R = ctx.download(dR, (n, n))
    GQ = _gram_all(ctx, info, dQ, m, n)
    GA = _gram_all(ctx, info, dA, m, n)
    idx, Qs = _row_sample(ctx, dQ, m, n)
    As = A[idx]
    out["tsqr_orth_max"] = float(np.max(np.abs(GQ - eye)))
    out["tsqr_resid_rows"] = d.max_over_ranks(float(np.linalg.norm(As - Qs @ R) / np.linalg.norm(As)))
    out["tsqr_gram_resid"] = float(np.linalg.norm(GA - R.T @ R) / np.linalg.norm(GA))
    out["tsqr_diag_min"] = float(np.min(np.diag(R)))
    out["tsqr_tril_max"] = float(np.max(np.abs(np.tril(R, -1))))
    digests = d.allgather_object(hashlib.sha1(R.tobytes()).hexdigest())
    out["tsqr_R_bitwise_replicated"] = len(set(digests)) == 1
    _require(out["tsqr_orth_max"] <= 1e-12, "TSQR ||Q^T Q - I||_max", out["tsqr_orth_max"])
    _require(out["tsqr_resid_rows"] <= 1e-12, "TSQR ||A - Q R|| / ||A|| (row sample, max over ranks)", out["tsqr_resid_rows"])
    _require(out["tsqr_gram_resid"] <= 1e-12, "TSQR ||A^T A - R^T R|| / ||A^T A||", out["tsqr_gram_resid"])
    _require(out["tsqr_diag_min"] > 0 and out["tsqr_tril_max"] == 0.0, "TSQR diag(R) > 0, tril(R) == 0", (out["tsqr_diag_min"], out["tsqr_tril_max"]))
    _require(out["tsqr_R_bitwise_replicated"], "TSQR R identical on every rank", digests)
    # ---- SVD via the Gram route
    s, Vt = ctx.download(ds, (n,)), ctx.download(dVt, (n, n))
    GU = _gram_all(ctx, info, dU, m, n)
    idx, Us = _row_sample(ctx, dU, m, n)
    As = A[idx]
    sR = np.linalg.svd(R, compute_uv=False)
    out["svd_U_orth_max"] = float(np.max(np.abs(GU - eye)))
    out["svd_V_orth_max"] = float(np.max(np.abs(Vt @ Vt.T - eye)))
    out["svd_resid_rows"] = d.max_over_ranks(float(np.linalg.norm(As - (Us * s) @ Vt) / np.linalg.norm(As)))
    out["svd_gram_resid"] = float(np.linalg.norm(GA - (Vt.T * s ** 2) @ Vt) / np.linalg.norm(GA))
    out["svd_s_vs_tsqr_R_rel"] = float(np.max(np.abs(s - sR) / sR))
    out["svd_s_descending"] = bool(np.all(np.diff(s) <= 0))
    digests = d.allgather_object(hashlib.sha1(s.tobytes() + Vt.tobytes()).hexdigest())
    out["svd_sVt_bitwise_replicated"] = len(set(digests)) == 1
    _require(out["svd_U_orth_max"] <= 1e-12, "SVD ||U^T U - I||_max", out["svd_U_orth_max"])
    _require(out["svd_V_orth_max"] <= 1e-12, "SVD ||V^T V - I||_max", out["svd_V_orth_max"])
    _require(out["svd_resid_rows"] <= 1e-12, "SVD ||A - U S V^T|| / ||A|| (row sample, max over ranks)", out["svd_resid_rows"])
    _require(out["svd_gram_resid"] <= 1e-12, "SVD ||A^T A - V S^2 V^T|| / ||A^T A||", out["svd_gram_resid"])
    _require(out["svd_s_vs_tsqr_R_rel"] <= 1e-10, "singular values: A^T A route vs np.linalg.svd(R_tsqr), relative", out["svd_s_vs_tsqr_R_rel"])
    _require(out["svd_s_descending"] and out["svd_sVt_bitwise_replicated"], "s descending / (s, Vt) identical on every rank", digests)
    out["tolerances"] = "orth <= 1e-12, residual <= 1e-12, singular values <= 1e-10 relative (BASELINE.json north_star)"
    return out


# ----------------------------------------------------------------------------- secondary configs
def run_extras(ctx, d, info, peaks):
    import linalg_b200 as lb  # noqa: F401

    out = {}
    dfma, dmma = ctx.probe(0), ctx.probe(1)
    out["fp64_peaks"] = {"dfma_tflops": dfma, "dmma_tflops": dmma, "copy_kernel_gbs": ctx.probe(2),
                         "how": "lq_probe micro-benchmarks in this run (MEASURED_PEAKS.json has no FP64 figure)"}
    peak64 = max(dfma, dmma)

    # ---- cfg3: batched Householder least squares, 2^16 systems of 256x64, 16 RHS (per GPU)
    nsys, m, n, k = 1 << 16, 256, 64, 16
    uniq = 1 << 11
    A = np.random.default_rng(3 + info.rank).standard_normal((uniq, m, n))
    B = np.random.default_rng(4 + info.rank).standard_normal((uniq, m, k))
    dA, dB = tile_to_device(ctx, A, nsys // uniq), tile_to_device(ctx, B, nsys // uniq)
    dX = ctx.alloc(8 * nsys * n * k)

    def check_lstsq(tag):
        # the LAST `uniq` systems of the timed batch against LAPACK (np.linalg.lstsq), 1e-10 relative per system
        # (north star: least-squares results to 1e-10), plus the normal equations A^T (A x - b) = 0
        nchk = 256
        X = np.empty((nchk, n, k))
        ctx.call("lq_memcpy_d2h", X.ctypes.data, dX.ptr + 8 * (nsys - nchk) * n * k, X.nbytes)
        ctx.sync()
        worst, worst_ne = 0.0, 0.0
        for i in range(nchk):
            Ai, Bi = A[uniq - nchk + i], B[uniq - nchk + i]
            Xo = np.linalg.lstsq(Ai, Bi, rcond=None)[0]
            worst = max(worst, float(np.max(np.abs(X[i] - Xo)) / np.max(np.abs(Xo))))
            worst_ne = max(worst_ne, float(np.linalg.norm(Ai.T @ (Ai @ X[i] - Bi)) / (np.linalg.norm(Ai) ** 2 * np.linalg.norm(X[i]))))
        _require(worst <= 1e-10, f"{tag}: max relative error vs np.linalg.lstsq over {nchk} systems", worst)
        _require(worst_ne <= 1e-13, f"{tag}: normal-equations residual", worst_ne)
        return {"systems_checked": nchk, "max_rel_err_vs_lapack": worst, "normal_eq_resid": worst_ne}

    ms = timed(ctx, lambda: ctx.call("lq_lstsq_householder_batched_dev", dA.ptr, dB.ptr, nsys, m, n, k, dX.ptr), 5, 3)
    t = d.max_over_ranks(statistics.mean(ms)) * 1e-3
    flops = 2905429.0
    out["cfg3_lstsq_hh_256x64x16"] = {
        "systems_per_s": info.world * nsys / t, "ms": t * 1e3, "gflops": info.world * nsys * flops / t / 1e9,
        "fp64_frac": nsys * flops / t / 1e12 / peak64, "hbm_frac": nsys * 172032 / t / 1e9 / peaks["hbm_gbs"],
        "parity": check_lstsq("cfg3 householder least squares")}
    dI = ctx.alloc(4 * nsys)
    ctx.call("lq_memset", dX.ptr, 0, 8 * nsys * n * k)
    ms = timed(ctx, lambda: ctx.call("lq_lstsq_mgs_batched_dev", dA.ptr, dB.ptr, nsys, m, n, k, dX.ptr, dI.ptr), 3, 2)
    t = d.max_over_ranks(statistics.mean(ms)) * 1e-3
    out["cfg3_lstsq_mgs_256x64x16"] = {"systems_per_s": info.world * nsys / t, "ms": t * 1e3,
                                       "fp64_frac": nsys * flops / t / 1e12 / peak64,
                                       "parity": check_lstsq("cfg3 MGS least squares")}
    for b in (dA, dB, dX, dI):
        b.free()

    # ---- cfg1 / cfg4: single-matrix blocked Householder (replicas only: every rank runs its own copy)
    for nn, reps in ((256, 20), (8192, 3)):
        A = np.random.default_rng(5).standard_normal((nn, nn))
        dA, dQ, dR = ctx.upload(A), ctx.alloc(A.nbytes), ctx.alloc(A.nbytes)
        l0 = ctx.launches()
        ms = timed(ctx, lambda: ctx.call("lq_householder_qr_dev", dA.ptr, nn, nn, dQ.ptr, dR.ptr), reps, 2, flush=(nn == 256))
        lpc = (ctx.launches() - l0) // (reps + 2)
        t = min(ms) * 1e-3
        fqr = 8.0 / 3.0 * nn ** 3
        # checked result: randomised invariants in O(n^2) host work (8 probe vectors) + exact structure of R
        Qh, Rh = ctx.download(dQ, (nn, nn)), ctx.download(dR, (nn, nn))
        Xp = np.random.default_rng(50).standard_normal((nn, 8))
        resid = float(np.linalg.norm(A @ Xp - Qh @ (Rh @ Xp)) / (np.linalg.norm(A) * np.linalg.norm(Xp) / np.sqrt(nn)))
        orth = float(np.linalg.norm(Qh.T @ (Qh @ Xp) - Xp) / np.linalg.norm(Xp))
        tril = float(np.max(np.abs(np.tril(Rh, -1))))
        # sign convention of linalg/qr.py:82-86: R[j, j] = -copysign(||x||, x0); for column 0, x0 = A[0, 0]
        sign0 = bool(np.sign(Rh[0, 0]) == -np.sign(A[0, 0])) and abs(abs(Rh[0, 0]) - np.linalg.norm(A[:, 0])) <= 1e-12 * np.linalg.norm(A[:, 0])
        _require(resid <= 1e-12 and orth <= 1e-12 and tril == 0.0 and sign0, f"blocked householder_qr {nn}^2 (resid, orth, tril, sign)", (resid, orth, tril, sign0))
        out[f"blocked_hh_{nn}"] = {"ms_best": t * 1e3, "ms_mean": statistics.mean(ms), "tflops_FQR": fqr / t / 1e12,
                                   "fp64_frac": fqr / t / 1e12 / peak64, "launches_per_call": int(lpc), "replicas": info.world,
                                   "parity": {"probe_resid": resid, "probe_orth": orth, "tril_max": tril, "r00_sign_and_norm": sign0}}
        del Qh, Rh
        for b in (dA, dQ, dR):
            b.free()

    # ---- cfg5: tall-skinny 2^20 x 128 rows per GPU, row-sharded with NCCL when N > 1 (weak), then 2^23 rows in total (strong)
    n = 128
    if info.world > 1:
        d.init_comm(ctx, info)
    sh = "_sharded" if info.world > 1 else ""
    for tag, m in (("", 1 << 20), ("_strong_8Mx128", (1 << 23) // info.world)):
        A = np.random.default_rng(6 + 1000 * info.rank).standard_normal((m, n))
        dA, dU, dQ, dR = ctx.upload(A), ctx.alloc(A.nbytes), ctx.alloc(A.nbytes), ctx.alloc(8 * n * n)
        ds, dVt = ctx.alloc(8 * n), ctx.alloc(8 * n * n)
        rk = C.c_int(0)
        ms = timed(ctx, lambda: ctx.call("lq_svd_gram" + sh + "_dev", dA.ptr, m, n, C.c_double(1e-12), dU.ptr, ds.ptr, dVt.ptr, C.byref(rk)), 5, 2)
        t = d.max_over_ranks(statistics.mean(ms)) * 1e-3
        f_svd = 3.0 * m * n * n            # Gram as a symmetric rank-k update (m n^2, SURVEY.md 8d) + U = A V S^-1 (2 m n^2)
        out["cfg5_svd_gram" + tag] = {"rows_total": m * info.world, "rows_per_gpu": m, "ms": t * 1e3, "gflops": info.world * f_svd / t / 1e9,
                                      "fp64_frac": f_svd / t / 1e12 / peak64, "rank": rk.value,
                                      "collective": "ncclAllReduce 128x128 f64" if info.world > 1 else None}
        ms = timed(ctx, lambda: ctx.call("lq_tsqr" + sh + "_dev", dA.ptr, m, n, dQ.ptr, dR.ptr), 5, 2)
        t = d.max_over_ranks(statistics.mean(ms)) * 1e-3
        executed = 6.0 * m * n * n      # CholeskyQR2: two SYRK Gram products (m n^2 each) + two A R^-1 products (2 m n^2 each)
        algorithmic = 4.0 * m * n * n   # Householder-equivalent: factor (2 m n^2) + explicit Q (2 m n^2)
        out["cfg5_tsqr" + tag] = {"rows_total": m * info.world, "rows_per_gpu": m, "ms": t * 1e3,
                                  "gflops_householder_equiv": info.world * algorithmic / t / 1e9,
                                  "fp64_frac_algorithmic": algorithmic / t / 1e12 / peak64,
                                  "executed_tflops_per_gpu": executed / t / 1e12, "fp64_frac_executed": executed / t / 1e12 / peak64,
                                  "hbm_frac": 2.0 * A.nbytes / t / 1e9 / peaks["hbm_gbs"],
                                  "collective": "2 x ncclAllReduce 128x128 f64 (Gram matrices)" if info.world > 1 else None}
        out["cfg5_parity" + tag] = check_cfg5(ctx, d, info, A, dA, dQ, dR, dU, ds, dVt, m, n)
        for b in (dA, dU, dQ, dR, ds, dVt):
            b.free()
        del A
    return out


if __name__ == "__main__":
    sys.exit(main())

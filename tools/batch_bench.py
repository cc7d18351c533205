"""Throughput of the batched solve (b200lp_solve_batch_*) on many small LPs of one shape.

For every workload: LPs/s and pivots/s of the batch kernel alone (CUDA events) and of the whole call (host clock
around the synchronised call, uploads and read-back included); a sequential loop of single solve() calls with the
memory cache on, and the CPU oracle, over a fixed subset, both as measured per-LP times.  Klee-Minty 20 through the
single-LP tiny kernel (simplex_tiny) is timed in the same process as a regression check of the shared pivot loop.

    python tools/batch_bench.py --out profiles/r03_batch_bench.json --repeats 2
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import oracle  # noqa: E402
import simplex_method_gpu_b200 as lp  # noqa: E402

MAX_ITER = 1 << 22          # Klee-Minty 20 through simplex_tiny
LP_MAX_ITER = 10000         # per LP of a batch: a few fp32 LPs cycle on degenerate vertices, the cap ends them


def gpu_info() -> dict:
    info = {}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,power.max_limit,clocks.max.sm",
                              "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=30).stdout
        name, pl, pmax, clk = [s.strip() for s in out.strip().split(",")]
        info.update(gpu=name, power_limit=pl, power_max_limit=pmax, max_sm_clock=clk)
    except Exception as e:                      # the numbers are still valid, the label is missing
        info["gpu_query_error"] = repr(e)
    return info


def dense_batch(batch, m, n, dt, seed0):
    """batch seeded dense LPs (oracle.gen_dense numbers), every LP column-major: returns A as (batch, m, n) views."""
    buf = np.empty((batch, n, m), dt)          # buf[k] is LP k's column-major m x n matrix
    b = np.empty((batch, m), dt)
    c = np.empty((batch, n), dt)
    for k in range(batch):
        oracle.gen_dense_into(buf[k].ctypes.data, b[k].ctypes.data, c[k].ctypes.data, m, n, seed0 + k, dt)
    return buf.transpose(0, 2, 1), b, c


def km_batch(batch, d):
    A0, b0, c0 = oracle.gen_klee_minty(d)
    m, n = A0.shape
    buf = np.empty((batch, n, m))
    buf[:] = A0.T
    return buf.transpose(0, 2, 1), np.tile(b0, (batch, 1)), np.tile(c0, (batch, 1))


def run_workload(name, A, b, c, eps, subset, repeats, max_iter=LP_MAX_ITER):
    batch, m, n = A.shape
    dt = A.dtype
    warm = min(batch, 512)
    lp.solve_batch(A[:warm], b[:warm], c[:warm], eps=eps, max_iter=max_iter, want_y=False)      # warm-up
    reps = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        bs = lp.solve_batch(A, b, c, eps=eps, max_iter=max_iter, want_y=False)
        wall = time.perf_counter() - t0
        piv = int(bs.pivots.sum())
        reps.append(dict(kernel_ms=bs.ms_solve, upload_ms=bs.ms_upload, download_ms=bs.ms_download, call_ms=wall * 1e3,
                         kernel_lps_per_s=batch / (bs.ms_solve * 1e-3), kernel_pivots_per_s=piv / (bs.ms_solve * 1e-3),
                         call_lps_per_s=batch / wall, call_pivots_per_s=piv / wall, kernel_launches=bs.kernel_launches))
    statuses = {int(s): int((bs.status == s).sum()) for s in np.unique(bs.status)}
    idx = np.arange(subset)
    sub_piv = int(bs.pivots[idx].sum())
    lp.set_memory_cache(True)
    lp.solve(A[0], b[0], c[0], eps=eps, max_iter=max_iter)                                        # warm-up
    seq = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        for k in idx:
            s = lp.solve(A[k], b[k], c[k], eps=eps, max_iter=max_iter)
            assert s.pivots == bs.pivots[k] and s.z == bs.z[k], (name, k)          # same bits as the batch
        seq.append((time.perf_counter() - t0) / subset * 1e3)
    lp.set_memory_cache(False)
    t0 = time.perf_counter()
    for k in idx:
        r = oracle.solve(np.asfortranarray(A[k]), b[k], c[k], eps=eps, max_iter=max_iter, order=1)
        assert r.pivots == bs.pivots[k] and r.z == bs.z[k], (name, k)
    ora = (time.perf_counter() - t0) / subset * 1e3
    out = dict(name=name, batch=batch, m=m, n=n, dtype=np.dtype(dt).name, eps=eps, max_iter=max_iter, pivots_total=int(bs.pivots.sum()),
               pivots_mean=float(bs.pivots.mean()), pivots_max=int(bs.pivots.max()), statuses=statuses, repeats=reps,
               subset=subset, subset_pivots=sub_piv, sequential_solve_ms_per_lp=seq, oracle_ms_per_lp=ora)
    r0 = reps[0]
    print(f"{name}: kernel {r0['kernel_lps_per_s']:.4g} LPs/s {r0['kernel_pivots_per_s']:.4g} piv/s | call "
          f"{r0['call_lps_per_s']:.4g} LPs/s | solve() loop {seq[0]:.3f} ms/LP | oracle {ora:.3f} ms/LP "
          f"| {[round(r['kernel_ms'], 2) for r in reps]} ms kernel", flush=True)
    return out


def km20_tiny(repeats):
    A, b, c = oracle.gen_klee_minty(20)
    lp.solve(A, b, c, eps=1e-4, max_iter=1 << 10)                                                  # warm-up
    us = []
    for _ in range(repeats):
        s = lp.solve(A, b, c, eps=1e-4, max_iter=MAX_ITER, trace_cap=1)
        assert s.pivots == 2 ** 20 - 1 and s.z == 5.0 ** 20
        us.append(s.ms_solve * 1e3 / s.pivots)
    print(f"Klee-Minty 20 (simplex_tiny): {us} us/pivot", flush=True)
    return dict(pivots=2 ** 20 - 1, us_per_pivot=us)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="JSON file to write")
    ap.add_argument("--repeats", type=int, default=2)
    ap.add_argument("--scale", type=float, default=1.0, help="shrink the batches (quick checks)")
    a = ap.parse_args()
    oracle.build()
    sc = lambda k: max(1, int(k * a.scale))
    res = dict(info=gpu_info(), workloads=[])
    res["km20_simplex_tiny"] = km20_tiny(a.repeats)
    A, b, c = dense_batch(sc(100000), 32, 96, np.float64, 1)
    res["workloads"].append(run_workload("dense_m32_n96_f64", A, b, c, 1e-9, min(1000, sc(100000)), a.repeats))
    A, b, c = dense_batch(sc(10000), 64, 192, np.float64, 200001)
    res["workloads"].append(run_workload("dense_m64_n192_f64", A, b, c, 1e-9, min(1000, sc(10000)), a.repeats))
    A, b, c = dense_batch(sc(10000), 128, 256, np.float32, 300001)
    res["workloads"].append(run_workload("dense_m128_n256_f32", A, b, c, 1e-4, min(1000, sc(10000)), a.repeats))
    A, b, c = km_batch(sc(1024), 14)
    res["workloads"].append(run_workload("klee_minty_d14", A, b, c, 1e-4, min(100, sc(1024)), a.repeats, 1 << 15))
    res["km20_simplex_tiny_after"] = km20_tiny(a.repeats)
    print(json.dumps(res["info"]))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

"""Throughput of the batched dual simplex and composite method (solve_batch with algorithm=1, with and without
cost_shift=1: simplex_tiny_batch_dual) on many small LPs of one shape.

Workloads: 100 000 covering LPs (dual_oracle.gen_covering's numbers: the dense generator with signs flipped,
m = 32, n = 96, fp64) and 10 000 dual_oracle.gen_general(..., "feasible") LPs (m = 32, n = 96, fp64, composite).
For each: the batch kernel's time (CUDA events) and the whole call's (host clock around the synchronised call,
uploads and read-back included); over a fixed subset, a loop of single solve() calls with the memory cache on (the
path these batches took before the batch kernel ran them: simplex_dual per LP) and the CPU reference dual_oracle,
as per-LP times.  Klee-Minty 20 through simplex_tiny is timed before and after, the regression check of the pivot
blocks the primal and dual loops share.

    python tools/batch_dual_bench.py --out profiles/r06_batch_dual_bench.json --repeats 2
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import dual_oracle  # noqa: E402
import oracle  # noqa: E402
import simplex_method_gpu_b200 as lp  # noqa: E402
from batch_bench import dense_batch, gpu_info, km20_tiny  # noqa: E402

LP_MAX_ITER = 10000
EPS = 1e-9


def covering_batch(batch, m, n, seed0):
    """gen_covering(m, n, seed0 + k) for every k, built from the dense generator in place"""
    A, b, c = dense_batch(batch, m, n, np.float64, seed0)
    ns = n - m
    A[:, :, :ns] *= -1.0
    c *= -1.0
    c[:, ns:] = 0.0                                # +0, as gen_covering
    return A, -b, c


def general_batch(batch, m, n, seed0):
    probs = [dual_oracle.gen_general(m, n, seed0 + k, "feasible") for k in range(batch)]
    return np.stack([p[0] for p in probs]), np.stack([p[1] for p in probs]), np.stack([p[2] for p in probs])


def run_workload(name, A, b, c, subset, repeats, **opts):
    batch, m, n = A.shape
    warm = min(batch, 512)
    lp.solve_batch(A[:warm], b[:warm], c[:warm], eps=EPS, max_iter=LP_MAX_ITER, want_y=False, algorithm=1, **opts)
    reps = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        bs = lp.solve_batch(A, b, c, eps=EPS, max_iter=LP_MAX_ITER, want_y=False, algorithm=1, **opts)
        wall = time.perf_counter() - t0
        piv = int(bs.pivots.sum())
        reps.append(dict(kernel_ms=bs.ms_solve, upload_ms=bs.ms_upload, download_ms=bs.ms_download, call_ms=wall * 1e3,
                         kernel_lps_per_s=batch / (bs.ms_solve * 1e-3), kernel_pivots_per_s=piv / (bs.ms_solve * 1e-3),
                         call_lps_per_s=batch / wall, call_pivots_per_s=piv / wall, kernel_launches=bs.kernel_launches))
    statuses = {int(s): int((bs.status == s).sum()) for s in np.unique(bs.status)}
    idx = np.arange(subset)
    lp.set_memory_cache(True)
    lp.solve(A[0], b[0], c[0], eps=EPS, max_iter=LP_MAX_ITER, algorithm=1, **opts)                      # warm-up
    seq = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        for k in idx:
            s = lp.solve(A[k], b[k], c[k], eps=EPS, max_iter=LP_MAX_ITER, algorithm=1, **opts)
            assert s.pivots == bs.pivots[k] and s.z == bs.z[k], (name, k)          # same bits as the batch
        seq.append((time.perf_counter() - t0) / subset * 1e3)
    lp.set_memory_cache(False)
    t0 = time.perf_counter()
    for k in idx:
        r = dual_oracle.solve(np.asfortranarray(A[k]), b[k], c[k], eps=EPS, max_iter=LP_MAX_ITER, order=1,
                              cost_shift=opts.get("cost_shift", 0))
        assert r.pivots == bs.pivots[k] and r.z == bs.z[k], (name, k)
    ora = (time.perf_counter() - t0) / subset * 1e3
    out = dict(name=name, batch=batch, m=m, n=n, dtype="float64", eps=EPS, max_iter=LP_MAX_ITER, options=opts,
               pivots_total=int(bs.pivots.sum()), pivots_mean=float(bs.pivots.mean()), pivots_max=int(bs.pivots.max()),
               statuses=statuses, repeats=reps, subset=subset, subset_pivots=int(bs.pivots[idx].sum()),
               sequential_solve_ms_per_lp=seq, oracle_ms_per_lp=ora)
    r0 = reps[-1]
    print(f"{name}: kernel {r0['kernel_ms']:.2f} ms = {r0['kernel_lps_per_s']:.4g} LPs/s {r0['kernel_pivots_per_s']:.4g} piv/s"
          f" | call {r0['call_ms']:.1f} ms = {r0['call_lps_per_s']:.4g} LPs/s | solve() loop {seq[-1]:.3f} ms/LP"
          f" | dual_oracle {ora:.3f} ms/LP", flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="JSON file to write")
    ap.add_argument("--repeats", type=int, default=2)
    ap.add_argument("--scale", type=float, default=1.0, help="shrink the batches (quick checks)")
    a = ap.parse_args()
    oracle.build()
    dual_oracle.build()
    sc = lambda k: max(1, int(k * a.scale))
    res = dict(info=gpu_info(), workloads=[])
    res["km20_simplex_tiny"] = km20_tiny(a.repeats)
    A, b, c = covering_batch(sc(100000), 32, 96, 1)
    res["workloads"].append(run_workload("covering_m32_n96_f64_dual", A, b, c, min(500, sc(100000)), a.repeats))
    del A, b, c
    A, b, c = general_batch(sc(10000), 32, 96, 1)
    res["workloads"].append(run_workload("general_feasible_m32_n96_f64_composite", A, b, c, min(500, sc(10000)),
                                         a.repeats, cost_shift=1))
    res["km20_simplex_tiny_after"] = km20_tiny(a.repeats)
    print(json.dumps(res["info"]))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

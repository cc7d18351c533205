"""Composite method (options.algorithm = 1, cost_shift = 1) on the feasible family of dual_oracle.gen_general (mixed-sign
b and c: the slack basis is neither primal nor dual feasible), fp64, one GPU.

For m = 1024 / n = 2048 and m = 8192 / n = 16384: time to optimal, and where it goes.  One run untimed by the
profiler (wall clock of b200lp_run and the engine's own device time ms_solve), then b200lp_reset and the same run
under torch.profiler (CUDA kernels only), whose kernel durations split it into
  shift      k_cost_shift
  phase 1    simplex_dual (pivots and us/pivot from the phase information)
  hand-over  the flush of the pending update (k_update_ftran), k_gather_cb, k_btran_vec, k_copy, k_objective
  phase 2    the primal loop kernel (simplex_resident or simplex_persistent; pivots and us/pivot)
Both runs are checked to end in the same optimum.  At m = 1024 also HiGHS' dual simplex (scipy 'highs-ds') and the
CPU reference (dual_oracle, order 1, OpenMP) to optimal on the same LP.

    python tools/composite_bench.py --out profiles/r05_composite_bench.json
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

import dual_oracle  # noqa: E402
import simplex_method_gpu_b200 as lp  # noqa: E402

EPS = 1e-9
SEED = 1
HANDOVER = ("k_update_ftran", "k_gather_cb", "k_btran_vec", "k_copy", "k_objective")
PHASE2 = ("simplex_persistent", "simplex_resident", "simplex_tiny")


def gpu_info() -> dict:
    import subprocess
    info = {}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                              "-i", "0"], capture_output=True, text=True, timeout=30).stdout
        name, pl, clk = [s.strip() for s in out.strip().split(",")]
        info.update(gpu=name, power_limit=pl, max_sm_clock=clk)
    except Exception as e:                      # the numbers are still valid, the label is missing
        info["gpu_query_error"] = repr(e)
    return info


def kernel_split(prof) -> dict:
    """device time (us) per part of the run from the profiler's kernel records"""
    out = {"shift": 0.0, "phase1": 0.0, "handover": 0.0, "phase2": 0.0, "other": 0.0}
    kernels = {}
    for ev in prof.events():
        if ev.device_type.name != "CUDA":
            continue
        us = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
        name = ev.name
        kernels[name] = kernels.get(name, 0.0) + us
        if "k_cost_shift" in name:
            out["shift"] += us
        elif "simplex_dual" in name:
            out["phase1"] += us
        elif any(k in name for k in HANDOVER):
            out["handover"] += us
        elif any(k in name for k in PHASE2):
            out["phase2"] += us
        else:
            out["other"] += us
    out["kernels"] = {k: round(v, 1) for k, v in sorted(kernels.items(), key=lambda kv: -kv[1])[:12]}
    return out


def arm(m: int, n: int, max_iter: int) -> dict:
    import torch
    from torch.profiler import ProfilerActivity, profile
    A, b, c = dual_oracle.gen_general(m, n, SEED, "feasible")
    rec = {"m": m, "n": n, "seed": SEED, "eps": EPS}
    with lp.Engine(m, n, dtype=np.float64, eps=EPS, max_iter=max_iter, algorithm=1, cost_shift=1) as e:
        t = time.perf_counter()
        e.upload(A, b, c)
        rec["upload_s"] = time.perf_counter() - t
        t = time.perf_counter()
        r = e.run(max_iter)
        rec["wall_s"] = time.perf_counter() - t
        rec["ms_solve"] = r["ms_solve"]
        ph = e.phase_info()
        rec.update(status=r["status"].name, iterations=r["iterations"], pivots=r["pivots"], z=r["z"], **ph)
        x_b, b_ixs, y = e.download()
        e.reset()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            r2 = e.run(max_iter)
            torch.cuda.synchronize()
        assert (r2["pivots"], r2["z"]) == (r["pivots"], r["z"]), "profiled run differs"
    split = kernel_split(prof)
    p1, p2 = ph["phase1_pivots"], r["pivots"] - ph["phase1_pivots"]
    rec["split_us"] = {k: round(v, 1) for k, v in split.items() if k != "kernels"}
    rec["kernels_us"] = split["kernels"]
    rec["phase1_us_per_pivot"] = round(split["phase1"] / max(p1, 1), 2)
    rec["phase2_us_per_pivot"] = round(split["phase2"] / max(p2, 1), 2)
    x = np.zeros(n)
    x[b_ixs] = x_b
    rec["certificate"] = {"max_infeas": float(max(0.0, (A @ x - b).max(), -x.min())),
                          "min_reduced_cost": float((y @ A - c).min()),
                          "gap_rel": float(abs(c @ x - y @ b) / max(1.0, abs(c @ x)))}
    return rec, (A, b, c)


def cpu_arms(A, b, c) -> dict:
    from scipy.optimize import linprog
    m, n = A.shape
    ns = n - m
    out = {}
    t = time.perf_counter()
    h = linprog(-c[:ns], A_ub=A[:, :ns], b_ub=b, bounds=(0, None), method="highs-ds")
    out["highs_ds_s"] = time.perf_counter() - t
    out["highs_z"] = float(-h.fun) if h.status == 0 else None
    t = time.perf_counter()
    s = dual_oracle.solve(A, b, c, eps=EPS, max_iter=10 ** 7, order=1, cost_shift=1, trace_cap=1)
    out["cpu_oracle_s"] = time.perf_counter() - t
    out["cpu_oracle_threads"] = os.cpu_count()
    out["cpu_oracle_z"] = s.z
    out["cpu_oracle_pivots"] = s.pivots
    return out


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=None)
    ap.add_argument("--sizes", default="1024x2048,8192x16384")
    ap.add_argument("--max-iter", type=int, default=10 ** 6)
    args = ap.parse_args()
    res = {"bench": "composite", **gpu_info(), "arms": []}
    for k, s in enumerate(args.sizes.split(",")):
        m, n = (int(v) for v in s.split("x"))
        rec, lpdata = arm(m, n, args.max_iter)
        if m == 1024:
            rec.update(cpu_arms(*lpdata))
        res["arms"].append(rec)
        print(json.dumps(rec), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

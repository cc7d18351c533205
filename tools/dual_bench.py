"""Dual simplex (options.algorithm = 1) on covering LPs against the primal Dantzig loop on the dense LP of the same
shape, fp64, one GPU.

Covering LP = the dense generator's LP negated (dual_oracle.gen_covering): min c_s.x s.t. A_s x >= b_s, x >= 0,
slack basis dual feasible and primal infeasible.  Arms, alternated dual / primal in this one process, `--repeats`
times each:
  m = 1024 / n = 2048 and m = 8192 / n = 16384: the dual solved to optimality (pivots, seconds, us/pivot, GB/s from
      the Dantzig bytes formula 8 (2 m^2 + m (n - m)) against the 6550 GB/s copy roofline, a host-side duality
      certificate), the primal a window of the same number of pivots on the dense LP (us/pivot)
  m = 32768 / n = 65536: a window of 192 pivots of each (us/pivot)
plus HiGHS dual simplex (scipy 'highs-ds', one thread) time to optimal at m = 1024, the CPU baseline, and the phase
stamps of one dual window at m = 8192 (where the time of a pivot goes).

    python tools/dual_bench.py --out profiles/r04_dual_bench.json --repeats 2
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
from simplex_method_gpu_b200.solver import lpgen_dense_into  # noqa: E402
from simplex_method_gpu_b200 import capi  # noqa: E402

EPS = 1e-9
COPY_ROOFLINE_GBS = 6550.0      # measured HBM copy bandwidth of one B200 (profiles/r01_membw_probe.txt)
WINDOW = 192
PRIMAL_SEED = 1
COVER_SEED = 1


def gpu_info() -> dict:
    import subprocess
    info = {}
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,power.max_limit,clocks.max.sm",
                              "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=30).stdout
        name, pl, pmax, clk = [s.strip() for s in out.strip().split(",")]
        info.update(gpu=name, power_limit=pl, power_max_limit=pmax, max_sm_clock=clk)
    except Exception as e:                      # the numbers are still valid, the label is missing
        info["gpu_query_error"] = repr(e)
    return info


def bytes_per_pivot(m, n):
    return 8 * (2 * m * m + m * (n - m))


def covering_structural(m, n, seed):
    """A_s (negated, column-major m x (n - m)), b, c of the covering LP; the identity slack block is not stored (the
    engine is told to trust it, check_slack = 0), which keeps m = 32768 at 8.6 GB of host memory."""
    ns = n - m
    A = np.empty((m, ns), np.float64, order="F")
    b = np.empty(m)
    c = np.empty(n)
    lpgen_dense_into(A.ctypes.data, b.ctypes.data, c.ctypes.data, m, n, 0, ns, seed)
    np.negative(A, out=A)
    c = -c
    c[ns:] = 0.0
    return A, -b, c


def certificate(A_s, b, c, x_b, b_ixs, y):
    """primal residual of [A_s, I] x = b, min reduced cost y.a_j - c_j, relative gap |c.x - y.b| / |c.x|"""
    m, ns = A_s.shape
    n = ns + m
    x = np.zeros(n)
    x[b_ixs] = x_b
    res = A_s @ x[:ns] + x[ns:] - b
    e = np.concatenate([y @ A_s - c[:ns], y - c[ns:]])
    pz, dz = float(c @ x), float(y @ b)
    return dict(primal_residual_max=float(np.abs(res).max()), x_min=float(x.min()), min_reduced_cost=float(e.min()),
                primal_objective=pz, dual_objective=dz, relative_gap=abs(pz - dz) / max(1.0, abs(pz)))


def dual_arm(A_s, b, c, iters, cert):
    m, ns = A_s.shape
    n = ns + m
    with lp.Engine(m, n, dtype=np.float64, eps=EPS, max_iter=iters, algorithm=1, check_slack=0) as e:
        e.upload_raw(A_s.ctypes.data, b.ctypes.data, c.ctypes.data)
        r = e.run(iters)
        out = dict(status=r["status"].name, pivots=r["pivots"], iterations=r["iterations"], seconds=r["ms_solve"] * 1e-3,
                   us_per_pivot=r["ms_solve"] * 1e3 / max(1, r["pivots"]), z=r["z"], grid_ctas=e.grid_ctas)
        out["gbs"] = bytes_per_pivot(m, n) * r["pivots"] / (r["ms_solve"] * 1e-3) / 1e9
        out["share_of_copy_roofline"] = out["gbs"] / COPY_ROOFLINE_GBS
        if cert:
            x_b, b_ixs, y = e.download()
            out["certificate"] = certificate(A_s, b, c, x_b, b_ixs, y)
    return out


def primal_arm(m, n, pivots):
    with lp.Engine(m, n, dtype=np.float64, eps=EPS, max_iter=pivots) as e:
        e.generate_dense(PRIMAL_SEED)
        r = e.run(pivots)
        return dict(status=r["status"].name, pivots=r["pivots"], seconds=r["ms_solve"] * 1e-3,
                    us_per_pivot=r["ms_solve"] * 1e3 / max(1, r["pivots"]), grid_ctas=e.grid_ctas,
                    gbs=bytes_per_pivot(m, n) * r["pivots"] / (r["ms_solve"] * 1e-3) / 1e9)


def phase_profile(A_s, b, c, iters):
    """mean ns per interval of the dual loop's phase stamps over one window (stamps 0..8, see kernels.cuh)"""
    m, ns = A_s.shape
    with lp.Engine(m, ns + m, dtype=np.float64, eps=EPS, max_iter=iters, algorithm=1, check_slack=0,
                   profile=iters) as e:
        e.upload_raw(A_s.ctypes.data, b.ctypes.data, c.ctypes.data)
        e.run(iters)
        st = e.profile().astype(np.int64)[:, :9]
    names = ["leaving row + rho gather + barrier", "column pass (e, alpha_r)", "barrier + both argmins",
             "update + FTRAN", "barrier + alpha sums", "barrier + book1", "barrier", "book2 + leaving candidates"]
    full = st[np.all(st > 0, axis=1)]
    d = np.diff(full, axis=1)
    return {k: float(v) / 1e3 for k, v in zip(names, d.mean(axis=0))} | {"iterations_profiled": int(len(full))}


def highs_baseline(A_s, b, c):
    from scipy.optimize import linprog
    ns = A_s.shape[1]
    t0 = time.perf_counter()
    r = linprog(-c[:ns], A_ub=A_s, b_ub=b, bounds=(0, None), method="highs-ds", options={"presolve": False})
    dt = time.perf_counter() - t0
    return dict(seconds=dt, status=int(r.status), objective=float(-r.fun), iterations=int(getattr(r, "nit", -1)),
                threads=1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--repeats", type=int, default=2)
    ap.add_argument("--big", type=int, default=1, help="0: skip m = 32768")
    a = ap.parse_args()
    capi.lib()
    res = dict(info=gpu_info(), bytes_per_pivot="8 (2 m^2 + m (n - m))", copy_roofline_gbs=COPY_ROOFLINE_GBS,
               eps=EPS, arms=[])
    shapes = [(1024, 2048, 10 ** 6, True), (8192, 16384, 10 ** 6, True)]
    if a.big:
        shapes.append((32768, 65536, WINDOW, False))
    for m, n, iters, to_opt in shapes:
        A_s, b, c = covering_structural(m, n, COVER_SEED)
        dual_arm(A_s, b, c, 3, False)                       # warm-up of both arms at this shape
        primal_arm(m, n, 3)
        arm = dict(m=m, n=n, dual=[], primal=[])
        for _ in range(a.repeats):
            d = dual_arm(A_s, b, c, iters, to_opt)
            p = primal_arm(m, n, d["pivots"] if to_opt else WINDOW)
            arm["dual"].append(d)
            arm["primal"].append(p)
            print(f"m={m} n={n}: dual {d['status']} {d['pivots']} pivots {d['seconds']:.4f} s "
                  f"{d['us_per_pivot']:.2f} us/pivot {d['gbs']:.0f} GB/s | primal {p['us_per_pivot']:.2f} us/pivot "
                  f"({p['pivots']} pivots)", flush=True)
        du = [x["us_per_pivot"] for x in arm["dual"]]
        pu = [x["us_per_pivot"] for x in arm["primal"]]
        arm["dual_us_per_pivot_spread"] = [min(du), max(du)]
        arm["primal_us_per_pivot_spread"] = [min(pu), max(pu)]
        arm["dual_over_primal_us_per_pivot"] = float(np.median(du) / np.median(pu))
        if m == 1024:
            arm["highs_ds"] = highs_baseline(A_s, b, c)
            print(f"HiGHS dual simplex m={m}: {arm['highs_ds']['seconds']:.3f} s", flush=True)
        if m == 8192:
            arm["dual_phase_us"] = phase_profile(A_s, b, c, WINDOW)
            print(f"phases m={m}: {arm['dual_phase_us']}", flush=True)
        res["arms"].append(arm)
        del A_s
    print(json.dumps(res["info"]))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

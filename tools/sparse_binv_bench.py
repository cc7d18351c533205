"""Touched-column passes (b200lp_set_binv_sparse, Engine(binv_sparse=...)) against the dense passes, in one process on one GPU.

Windows from the slack basis on bench.py's LPs (dense, seed 1, eps 1e-9, fp64), the two arms alternated:
  C4 (m = 32768, n = 65536) 192-pivot windows and C3 (m = 8192, n = 16384) 1000-pivot windows, 3 warm-up windows
  per arm, then --pairs pairs; optionally (--tto) C3 Dantzig and C4 steepest edge from the slack basis to the optimum.
Reports per-pivot time (CUDA events on the engine's stream) with its spread, the phase stamps of one extra profiled
window per arm, |K| (distinct leaving rows since the reset) at the end of each window, and the bytes each arm moves
per pivot: dense 8 m (n - m) + 16 m^2, sparse 8 m (n - m) + 16 m |K| (mean |K| over the window's pivots; the O(m)
vectors and the chunk partials are left out of both).  Asserts that the arms agree on the trace digest and on the
bits of x_b, y and z.  Writes --out (profiles/r07_sparse_binv.json by default)."""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import simplex_method_gpu_b200 as lp  # noqa: E402

SEED, EPS = 1, 1e-9
NAMES = json.loads(lp.capi.lib().b200lp_profile_names().decode())["single"]


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm,clocks.mem"
    try:
        return subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True,
                              text=True, timeout=30).stdout.strip()
    except Exception as ex:   # the numbers below are still taken; the card is then unnamed
        return f"nvidia-smi unavailable: {ex}"


def mean_k(trace):
    """|K| after every pivot of a window from the slack basis, and its value at the end"""
    seen, ks = set(), []
    for q in trace[:, 1].tolist():
        seen.add(q)
        ks.append(len(seen))
    return (float(np.mean(ks)) if ks else 0.0), len(seen)


def window(eng, P):
    eng.reset()
    r = eng.run(P)
    tr = eng.trace(P)
    x_b, _, y = eng.download()
    return {"ms": r["ms_solve"], "pivots": r["pivots"], "z": r["z"], "trace": tr,
            "digest": hashlib.sha256(np.ascontiguousarray(tr, np.int32).tobytes()).hexdigest(),
            "xb": x_b.view(np.uint64).copy(), "y": y.view(np.uint64).copy()}


def phases(m, n, P):
    """median time of every stamp interval over one profiled window per arm (separate engines)"""
    out = {}
    for arm in (-1, 0):
        with lp.Engine(m, n, np.float64, eps=EPS, max_iter=1 << 40, binv_sparse=arm, profile=P) as e:
            e.generate_dense(SEED)
            e.run(4)
            e.reset()
            e.run(P)
            st = e.profile(P).astype(np.int64)
        d = np.diff(np.concatenate([st, np.roll(st[:, :1], -1, axis=0)], axis=1), axis=1)[:-1]
        res = {}
        for k, name in enumerate(NAMES):
            if name == "-":
                continue
            v = d[:, k]
            v = v[(v > 0) & (v < 10**9)]
            if len(v):
                res[name] = round(float(np.median(v)) / 1e3, 2)
        out["dense" if arm < 0 else "sparse"] = res
    return out


def windows(name, m, n, P, pairs):
    engs = {arm: lp.Engine(m, n, np.float64, eps=EPS, max_iter=1 << 40, binv_sparse=arm) for arm in (-1, 0)}
    for e in engs.values():
        e.generate_dense(SEED)
    for _ in range(3):
        for e in engs.values():
            window(e, P)
    rows = {-1: [], 0: []}
    for _ in range(pairs):
        for arm in (-1, 0):
            rows[arm].append(window(engs[arm], P))
    for e in engs.values():
        e.close()
    d0, s0 = rows[-1][-1], rows[0][-1]
    assert d0["digest"] == s0["digest"], name
    assert np.array_equal(d0["xb"], s0["xb"]) and np.array_equal(d0["y"], s0["y"]) and d0["z"] == s0["z"], name
    assert all(r["digest"] == d0["digest"] for r in rows[-1] + rows[0]), name
    kmean, kend = mean_k(s0["trace"])
    out = {"workload": f"{name}: m={m} n={n} fp64, {P}-pivot windows from the slack basis", "pairs": pairs,
           "trace_sha256": d0["digest"], "z_after_window": d0["z"], "K_end": kend, "K_mean": kmean}
    dense_b = 8 * m * (n - m) + 16 * m * m
    sparse_b = 8 * m * (n - m) + 16 * m * kmean
    for arm, key, byt in ((-1, "dense", dense_b), (0, "sparse", sparse_b)):
        us = np.array([r["ms"] * 1e3 / r["pivots"] for r in rows[arm]])
        out[key] = {"us_per_pivot": [round(float(x), 1) for x in us], "median": float(np.median(us)),
                    "min": float(us.min()), "max": float(us.max()), "spread_pct": float((us.max() - us.min()) / np.median(us) * 100),
                    "bytes_per_pivot": float(byt), "TBps_on_those_bytes": float(byt / (np.median(us) * 1e-6) / 1e12)}
    out["speedup_median"] = out["dense"]["median"] / out["sparse"]["median"]
    out["phases_us_median"] = phases(m, n, P)
    return out


def to_optimal(name, m, n, rule):
    out = {"workload": f"{name}: m={m} n={n} fp64, slack basis to the optimum",
           "pricing_rule": "steepest edge" if rule else "Dantzig"}
    got = {}
    for arm in (-1, 0):
        with lp.Engine(m, n, np.float64, eps=EPS, max_iter=1 << 40, binv_sparse=arm, pricing_rule=rule) as e:
            e.generate_dense(SEED)
            e.run(8)
            e.reset()
            r = e.run(1 << 40)
            x_b, _, y = e.download()
            kmean, kend = mean_k(e.trace(1 << 22))
            got[arm] = (r, x_b.view(np.uint64).copy(), y.view(np.uint64).copy())
            out["dense" if arm < 0 else "sparse"] = {"seconds": r["ms_solve"] * 1e-3, "pivots": int(r["pivots"]),
                                                    "z": r["z"], "status": int(r["status"]), "K_end": kend, "K_mean": kmean}
    (rd, xd, yd), (rs, xs, ys) = got[-1], got[0]
    assert rd["pivots"] == rs["pivots"] and rd["z"] == rs["z"] and np.array_equal(xd, xs) and np.array_equal(yd, ys), name
    out["speedup"] = out["dense"]["seconds"] / out["sparse"]["seconds"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=5)
    ap.add_argument("--tto", action="store_true", help="also C3 Dantzig and C4 steepest edge to the optimum")
    ap.add_argument("--small", action="store_true", help="m = 2048 / 4096 instead of C3 / C4 (a rehearsal)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_sparse_binv.json"))
    a = ap.parse_args()
    c3, c4 = ((2048, 4096), (4096, 8192)) if a.small else ((8192, 16384), (32768, 65536))
    res = {"gpu_before": gpu_info(), "date": time.strftime("%Y-%m-%d %H:%M:%S")}
    res["C4"] = windows("C4", *c4, 192, a.pairs)
    print(json.dumps({"C4": {k: res["C4"][k] for k in ("speedup_median", "K_end")}}), flush=True)
    res["C3"] = windows("C3", *c3, 1000, a.pairs)
    print(json.dumps({"C3": {k: res["C3"][k] for k in ("speedup_median", "K_end")}}), flush=True)
    if a.tto:
        res["C3_dantzig_to_optimal"] = to_optimal("C3", *c3, 0)
        print(json.dumps({"C3 tto": res["C3_dantzig_to_optimal"]["speedup"]}), flush=True)
        res["C4_steepest_edge_to_optimal"] = to_optimal("C4", *c4, 1)
    res["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()

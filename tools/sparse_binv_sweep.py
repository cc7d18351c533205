"""Sweep of the touched-column passes against the dense ones over m and |K| (DESIGN.md 3h: where the auto setting of
b200lp_set_binv_sparse switches).

For every LP (bench.py's dense generator, seed 1, eps 1e-9, fp64, n = 2m) and pricing rule, the same solve runs twice
with phase stamps, once with every pass dense (binv_sparse = -1) and once with the sparse passes forced on
(binv_sparse = m: no threshold, no size gate).  Both arms make the same pivots, so iteration i has the same |K| (the
distinct leaving rows of pivots 0 .. i-1) in both, and the per-iteration times compare directly.  Reported per |K| bin:
the median time per iteration of the whole pivot, of the update + FTRAN + ratio phases (stamps 2 -> 5) and of
book1 + BTRAN (stamps 5 -> 6), for both arms.  C4 (m = 32768) runs a window of --c4-pivots Dantzig pivots instead of a
whole solve.  Writes --out (profiles/r08_sparse_binv_sweep.json by default)."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import simplex_method_gpu_b200 as lp  # noqa: E402

SEED, EPS = 1, 1e-9


def one(m, n, rule, arm, iters):
    with lp.Engine(m, n, np.float64, eps=EPS, max_iter=1 << 40, binv_sparse=arm, pricing_rule=rule, resident=-1,
                   profile=min(iters, 1 << 16)) as e:
        e.generate_dense(SEED)
        e.run(4)
        e.reset()
        r = e.run(iters)
        st = e.profile(1 << 16).astype(np.int64)
        tr = e.trace(1 << 22)
        grid = e.grid_ctas
    k = st.shape[0] - 1                                # the last iteration has no successor stamp
    total = st[1:k + 1, 0] - st[:k, 0]
    upd = st[:k, 5] - st[:k, 2]
    bt = st[:k, 6] - st[:k, 5]
    return r, tr, grid, np.stack([total, upd, bt], 1) / 1e3


def sweep(m, n, rule, iters):
    rd, trd, grid, td = one(m, n, rule, -1, iters)
    rs, trs, _, ts = one(m, n, rule, m, iters)
    assert rd["pivots"] == rs["pivots"] and rd["z"] == rs["z"] and np.array_equal(trd, trs), (m, rule)
    seen, kk = set(), []
    for q in trs[:, 1].tolist():
        kk.append(len(seen))
        seen.add(q)
    k = min(len(kk), td.shape[0], ts.shape[0])
    kk = np.array(kk[:k])
    td, ts = td[:k], ts[:k]
    edges = np.unique(np.linspace(0, kk.max() + 1, 9).astype(int))
    bins = []
    for lo, hi in zip(edges[:-1], edges[1:]):
        sel = (kk >= lo) & (kk < hi)
        if sel.sum() < 3:
            continue
        d, s = np.median(td[sel], 0), np.median(ts[sel], 0)
        bins.append({"K": [int(lo), int(hi)], "iterations": int(sel.sum()),
                     "dense_us": {"pivot": round(d[0], 2), "update_ftran_ratio": round(d[1], 2), "book1_btran": round(d[2], 2)},
                     "sparse_us": {"pivot": round(s[0], 2), "update_ftran_ratio": round(s[1], 2), "book1_btran": round(s[2], 2)},
                     "pivot_ratio_sparse_over_dense": round(s[0] / d[0], 3)})
    nslab = (m + 1023) // 1024
    return {"m": m, "n": n, "rule": "steepest edge" if rule else "Dantzig", "grid_ctas": grid, "pivots": int(rd["pivots"]),
            "K_end": len(seen), "sparse_items_max": nslab * ((m + 255) // 256),
            "solve_ms": {"dense": rd["ms_solve"], "sparse": rs["ms_solve"]}, "bins": bins}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1024,2048,3072,4096,8192")
    ap.add_argument("--c4-pivots", type=int, default=3000)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_sparse_binv_sweep.json"))
    a = ap.parse_args()
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    res = {"gpu": subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True,
                                 text=True).stdout.strip(), "runs": []}
    for m in [int(x) for x in a.sizes.split(",") if x]:
        for rule in (0, 1):
            r = sweep(m, 2 * m, rule, 1 << 40)
            res["runs"].append(r)
            print(json.dumps({k: r[k] for k in ("m", "rule", "pivots", "K_end", "solve_ms")}), flush=True)
    if a.c4_pivots > 0:
        r = sweep(32768, 65536, 0, a.c4_pivots)
        res["runs"].append(r)
        print(json.dumps({k: r[k] for k in ("m", "rule", "pivots", "K_end", "solve_ms")}), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()

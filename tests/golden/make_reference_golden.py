"""Generates tests/golden/reference.json: solver results on the LPs of tests/test_reference_gpu.py, which those
tests compare against where the reference's own v4 build (oracle/_ref) is absent.

    python tests/golden/make_reference_golden.py

The file's "source" field says where the results came from:
- "reference v4 build (oracle/_ref)" when that build is present for both float and double;
- otherwise "CPU oracle", the repository's C restatement of the reference loop (oracle/simplex_oracle.c).

The oracle is not the reference.  Where the reference build exists, the tests pin the oracle to it pivot for pivot.
Oracle results therefore stand in for the reference only where the pivot sequence cannot depend on summation
order.  So for random dense LPs this script refuses to write a near-tie (runner-up gap <= 1e-12).  Values that
depend on summation order, such as the last bits of x_b or an fp32 objective, differ from the reference's.  The
tests compare them within their stated tolerances.
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import oracle  # noqa: E402

TIE = 1e-12
USE_REF = oracle.ref_available(np.float64) and oracle.ref_available(np.float32)


def solve(A, b, c, eps, max_iter, exact=False):
    """exact: integer data whose ties are exact and broken by the lowest index whatever the summation order."""
    if USE_REF:
        return oracle.ref_solve(A, b, c, eps=eps, max_iter=max_iter)
    r = oracle.solve(A, b, c, eps=eps, max_iter=max_iter)
    if not exact and r.pivots and min(r.gap_p.min(), r.gap_q.min()) <= TIE:
        sys.exit("near-tie: the oracle's pivot sequence may differ from the reference's; not written")
    return r


def entry(r, head=None):
    k = len(r.trace_p) if head is None else head
    return {"status": int(r.status), "iterations": int(r.iterations), "pivots": int(r.pivots), "z": float(r.z),
            "trace_p": r.trace_p[:k].tolist(), "trace_q": r.trace_q[:k].tolist(),
            "x_b": [float(v) for v in r.x_b], "b_ixs": r.b_ixs.tolist()}


def main():
    out = {"source": "reference v4 build (oracle/_ref)" if USE_REF else
                     "CPU oracle (oracle/simplex_oracle.c); the reference build was not available"}
    out["dense_f64"] = {f"{m}x{n}_s{s}": entry(solve(*oracle.gen_dense(m, n, s), 1e-9, 1 << 20))
                        for m, n, s in [(64, 128, 1), (256, 512, 1), (300, 700, 2), (1024, 2048, 1), (64, 128, 5)]}
    out["dense_f32"] = {f"{m}x{n}_s{s}": entry(solve(*oracle.gen_dense(m, n, s, dtype=np.float32), 1e-4, 100000), head=8)
                        for m, n, s in [(64, 160, 2), (200, 456, 3), (64, 128, 5)]}
    out["klee_minty_10"] = entry(solve(*oracle.gen_klee_minty(10), 1e-4, 1 << 20, exact=True))
    out["assignment_16"] = entry(solve(*oracle.gen_assignment(16, 1)[:3], 1e-4, 1 << 20, exact=True))
    with open(os.path.join(HERE, "reference.json"), "w") as f:
        json.dump(out, f, indent=0)
    print("wrote", os.path.join(HERE, "reference.json"), "from", out["source"])


if __name__ == "__main__":
    main()

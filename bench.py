#!/usr/bin/env python
"""Benchmark of the hot path: pivots/s of the dense revised simplex loop on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
                    [--workload C2|C3|C4] [--pivots P] [--dump-outputs DIR]

A "step" is one window of P pivots of the loop at src/v4_cub_reduction.cu:286-359 on
a synthetic dense LP (oracle/lpgen_dense: A_s ~ U(0,1), b = (n_s/2)U(1,2),
c_s ~ U(0.5,1.5), slack block last).  Default workload = the configuration
BASELINE.json quotes its metric on: m=32768, n=65536, fp64 (fits one B200).

  value ..... pivots/s with the LP resident in HBM (CUDA events on the engine's stream); same number
              under device_loop, the like-for-like figure against the reference arm's device_loop
  e2e ....... pivots/s through b200lp_solve_f64() with pinned HOST buffers: per step the cudaMalloc
              of all device state, the H2D of the LP, the pivots, the D2H of the result and the
              cudaFree are inside the timed region (what the reference's solve() does per call,
              v4:245-271, 366-377); e2e_cached = the same with b200lp_set_memory_cache(1)
  trace_sha256  sha256 of the int32 (p, q) trace of the last window: the same hash must come out of
              every GPU count, of the reference arm and of tests/golden/trace_digests.json (CPU oracle)
  roofline .. algorithmic bytes per pivot 8*(2 m^2 + m (n-m)) / measured time, against
              the measured HBM copy bandwidth in MEASURED_PEAKS.json
  cpu_baseline  the CPU oracle (port of the reference loop) on the box's host cores,
              bounded sample, rank 0, N=1 only

--impl reference times the reference's own v4 CUDA solver (oracle/_ref, built from
/root/reference by oracle/make_ref.sh with the documented minimal patches) on the same
LP and window, host buffers pinned like the reference's own main() (v4:408-414); when that
library is unavailable it falls back to the CPU oracle port.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    "C2": dict(m=1024, n=2048, pivots=1000),
    "C3": dict(m=8192, n=16384, pivots=1000),
    "C4": dict(m=32768, n=65536, pivots=192),
}
SEED = 1
EPS = 1e-9


def config_for(name, m, n, P):
    """The `config` object: key for key the same in both arms and at every GPU count."""
    return {"workload": f"{name}: dense LP m={m} n={n} (n counts the slack block), seed {SEED}, "
                        f"window of {P} pivots per step from the slack basis",
            "m": m, "n": n, "pivots_per_step": P, "eps": EPS, "seed": SEED,
            "l2": "working set (A_N + B^-1) larger than L2, no flush needed" if bytes_per_pivot(m, n) > 2 * 126e6 else
                  "working set fits the 126 MB L2 (L2-resident; roofline fraction may exceed 1)"}


def trace_digest(trace):
    """sha256 over the little-endian int32 (p, q) rows of a pivot trace."""
    a = np.ascontiguousarray(np.asarray(trace, dtype=np.int32).reshape(-1, 2)).astype("<i4")
    return hashlib.sha256(a.tobytes()).hexdigest()


def golden_digest(name, P):
    """Digest of the same window from the CPU oracle (tests/golden/trace_digests.json), or None."""
    try:
        with open(os.path.join(ROOT, "tests", "golden", "trace_digests.json")) as f:
            w = json.load(f)[name]["windows"][str(P)]
        return w["trace_sha256"], w["z"]
    except Exception:
        return None, None


def parity_fields(name, P, trace, z):
    sha = trace_digest(trace)
    gold, gz = golden_digest(name, P)
    out = {"trace_sha256": sha, "trace_pivots": int(len(trace)), "z_after_window": float(z)}
    if gold is not None:
        out["trace_matches_golden"] = bool(sha == gold)
        out["z_rel_diff_vs_golden"] = abs(z - gz) / max(1.0, abs(gz))
    return out


def profiled_traffic(workload, pivots_per_launch):
    """dram__bytes_read.sum + dram__bytes_write.sum of the persistent kernel from the committed ncu capture
    (profiles/r01_traffic.json, written by tools/ncu_extract.py), scaled to this launch's pivot count."""
    try:
        name = "r02_traffic.json" if os.path.exists(os.path.join(ROOT, "profiles", "r02_traffic.json")) else "r01_traffic.json"
        with open(os.path.join(ROOT, "profiles", name)) as f:
            t = json.load(f)[workload]
        return t["dram_bytes_per_pivot"] * pivots_per_launch, t
    except Exception:
        return None, None


def time_to_optimal(name, wl, dev=0, rule=0):
    """Whole solve from the slack basis to the optimum on one GPU (the other half of BASELINE.json's metric).
    rule 0 = the reference's Dantzig rule (v4:288-302), 1 = steepest edge (options.pricing_rule, README.md:16-17)."""
    import simplex_method_gpu_b200 as lp
    m, n = wl["m"], wl["n"]
    eng = lp.Engine(m, n, np.float64, eps=EPS, max_iter=1 << 40, device=dev, pricing_rule=rule)
    eng.generate_dense(SEED)
    eng.run(8)                       # warm-up launch
    eng.reset()
    t0 = time.perf_counter()
    r = eng.run(1 << 40)
    wall = time.perf_counter() - t0
    x_b, b_ixs, y = eng.download()
    drift, scale = eng.check_basis()          # |B^-1 b - x_b| after all those rank-1 updates without a refactorisation
    bytes_pp = eng.bytes_per_pivot
    eng.close()
    bpp = bytes_pp
    out = {"workload": f"{name}: dense LP m={m} n={n}, seed {SEED}, slack basis to optimum",
           "pricing_rule": "steepest edge (Goldfarb-Reid recurrence)" if rule else "Dantzig (the reference's rule)",
           "status": int(r["status"]), "bytes_per_pivot": bpp,
           "achieved_GBps": bpp * r["pivots"] / (r["ms_solve"] * 1e-3) / 1e9,
           "basis_drift": {"max_abs_Binv_b_minus_x_b": drift, "max_abs_x_b": scale},
           "pivots": int(r["pivots"]), "iterations": int(r["iterations"]), "z": r["z"],
           "seconds": r["ms_solve"] * 1e-3, "wall_seconds": wall, "pivots_per_s": r["pivots"] / (r["ms_solve"] * 1e-3)}
    out["certificate"] = optimality_certificate(m, n, x_b, b_ixs, y, r["z"])
    return out


def klee_minty_20(dev=0):
    """BASELINE config 5a: the Klee-Minty cube of dimension 20 (m=20, n=40, all data exact integers < 2^53) —
    exactly 2^20 - 1 Dantzig pivots to the optimum 5^20, a pure latency test (simplex_tiny: one CTA, state in shared memory)."""
    import simplex_method_gpu_b200 as lp
    d = 20
    A = np.zeros((d, 2 * d), order="F")
    for i in range(d):
        for j in range(i):
            A[i, j] = 2.0 ** (i - j + 1)
        A[i, i] = 1.0
        A[i, d + i] = 1.0
    b = 5.0 ** np.arange(1, d + 1)
    c = np.concatenate([2.0 ** np.arange(d - 1, -1, -1), np.zeros(d)])
    with lp.Engine(d, 2 * d, np.float64, eps=1e-4, max_iter=1 << 40, device=dev) as e:
        e.upload(A, b, c)
        r = e.run(1 << 40)
    return {"workload": "Klee-Minty cube d=20 (m=20, n=40)", "status": int(r["status"]), "pivots": int(r["pivots"]),
            "expected_pivots": 2 ** d - 1, "z": r["z"], "z_exact": bool(r["z"] == 5.0 ** d), "seconds": r["ms_solve"] * 1e-3,
            "us_per_pivot": r["ms_solve"] * 1e3 / max(int(r["pivots"]), 1), "kernel": "simplex_tiny<double>"}


def optimality_certificate(m, n, x_b, b_ixs, y, z):
    """Solver-independent proof of optimality (GLPK is absent, HiGHS is too slow on a dense 8192 x 8192 LP):
    primal feasibility A_s x <= b, x >= 0, dual feasibility y >= 0, y'A_s >= c_s, and zero duality gap c'x = b'y,
    all evaluated on the host in fp64 from the engine's x_b / b_ixs / y and the regenerated LP."""
    import simplex_method_gpu_b200 as lp
    ns = n - m
    A = np.empty((m, ns), np.float64, order="F")
    b = np.empty(m, np.float64)
    c = np.empty(n, np.float64)
    lp.solver.lpgen_dense_into(A.ctypes.data, b.ctypes.data, c.ctypes.data, m, n, 0, ns, SEED)
    x = np.zeros(n)
    x[b_ixs] = x_b
    xs = x[:ns]
    primal_res = float(np.max(A @ xs - b))                 # <= 0 up to rounding
    dual_res = float(np.min(y @ A - c[:ns]))               # >= -eps: reduced costs of the structural columns
    cx, by = float(c[:ns] @ xs), float(b @ y)
    scale = max(1.0, abs(cx))
    return {"max_Ax_minus_b": primal_res, "min_x": float(x.min()), "min_y": float(y.min()),
            "min_reduced_cost": dual_res, "c_x": cx, "b_y": by, "rel_duality_gap": abs(cx - by) / scale,
            "rel_z_minus_c_x": abs(z - cx) / scale,
            "optimal_within": {"feasibility": 1e-7 * float(np.abs(b).max()), "eps": EPS, "gap": 1e-9},
            "holds": bool(primal_res <= 1e-7 * np.abs(b).max() and x.min() >= -1e-7 and y.min() >= -1e-7
                          and dual_res >= -1e-7 and abs(cx - by) <= 1e-9 * scale)}


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def bytes_per_pivot(m, n, itemsize=8):
    return itemsize * (2 * m * m + m * (n - m))


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """--dump-outputs: write each array as out_dir/<name>.npy in float64 (int32 indices are exact there), so that two
    builds can be compared output for output on the same seeded LP.  When the arrays exceed DUMP_BYTES together, each
    keeps the same share of its rows, chosen by a fixed seed."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: np.asarray(v, np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    for name, a in arrays.items():
        if total > DUMP_BYTES and len(a) > 1:
            keep = max(1, len(a) * DUMP_BYTES // total)
            a = a[np.sort(np.random.default_rng(SEED).choice(len(a), keep, replace=False))]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None
        self.t0 = self.t1 = None

    def mark_start(self):
        """Start of the timed region (the sampler itself is started earlier: nvidia-smi needs ~1 s to come up)."""
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def __exit__(self, *exc):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = self.rows
        if self.t0 is not None:
            t1 = self.t1 if self.t1 is not None else time.time()
            inside = [r for t, r in rows if self.t0 <= t <= t1 + 0.06]
            # a window shorter than the sampling period: take the samples that bracket it
            rows = inside if inside else [r for t, r in rows if self.t0 - 0.25 <= t <= t1 + 0.25]
        else:
            rows = [r for _, r in rows]
        for r in rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for nm, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------- our arm, one GPU

def run_b200_single(args, wl):
    import torch

    import simplex_method_gpu_b200 as lp
    m, n, P = wl["m"], wl["n"], args.pivots or wl["pivots"]
    dev = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(dev)

    # ---- device-resident throughput ("value"): LP generated in HBM, windows of P pivots
    eng = lp.Engine(m, n, np.float64, eps=EPS, max_iter=1 << 40, device=dev)
    eng.generate_dense(SEED)
    stream = torch.cuda.ExternalStream(eng.stream, device=dev)
    # every step: back to the slack basis (untimed), then a window of P pivots (timed)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    pivots_timed, launches, internal_ms = 0, 0, 0.0
    with ClockSampler(dev) as clk:
        for _ in range(args.warmup):
            eng.reset()
            r = eng.run(P)
        torch.cuda.synchronize()
        clk.mark_start()
        for a, b_ in ev:
            eng.reset()
            l0 = eng.run(0)["kernel_launches"]
            torch.cuda.synchronize()
            a.record(stream)
            eng.run_async(P)
            b_.record(stream)
            r = eng.wait()
            pivots_timed += r["pivots"]
            launches += r["kernel_launches"] - l0
            internal_ms += r["ms_solve"]
        torch.cuda.synchronize()
        clk.mark_end()
    step_ms = [a.elapsed_time(b_) for a, b_ in ev]
    total_ms = float(sum(step_ms))
    value = pivots_timed / (total_ms * 1e-3)
    status_after = int(r["status"])
    grid = eng.grid_ctas
    trace = eng.trace(P)
    parity = parity_fields(args.workload, P, trace, r["z"])
    if args.dump_outputs:
        x_b, b_ixs, y = eng.download()      # the state the last timed window left: what b200lp_download hands a caller
        dump_outputs(args.dump_outputs, {"x_b": x_b, "b_ixs": b_ixs, "y": y, "trace": trace, "z": [r["z"]]})
    eng.close()

    # ---- end to end through the C ABI with host buffers ("e2e")
    e2e = e2e_cached = None
    if not args.no_e2e:
        A_pin = torch.empty((n, m), dtype=torch.float64, pin_memory=True)    # column-major m x n
        b_pin = torch.empty(m, dtype=torch.float64, pin_memory=True)
        c_pin = torch.empty(n, dtype=torch.float64, pin_memory=True)
        A_np = A_pin.numpy().T                                                # Fortran-ordered view
        lp.solver.lpgen_dense_into(A_pin.data_ptr(), b_pin.data_ptr(), c_pin.data_ptr(), m, n, 0, n, SEED)
        def timed_calls(cached):
            # cached: a caller that solves one LP after another keeps the device buffers between calls
            # (b200lp_set_memory_cache); default / headline: like the reference, every call allocates and
            # frees all device state (v4:245-264, 370-377)
            lp.set_memory_cache(cached)
            times, piv, sol = [], 0, None
            for s_ in range(args.warmup + args.steps):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                sol = lp.solve(A_np, b_pin.numpy(), c_pin.numpy(), eps=EPS, max_iter=P, device=dev, trace_cap=P)
                torch.cuda.synchronize()
                dt = time.perf_counter() - t0
                if s_ >= args.warmup:
                    times.append(dt)
                    piv += sol.pivots
            lp.set_memory_cache(False)
            return {"value": piv / sum(times), "unit": "pivots/s", "ms_per_step": 1e3 * sum(times) / len(times),
                    "ms_per_step_each": [round(1e3 * t, 1) for t in times],
                    "value_at_median_step": (piv / len(times)) / float(np.median(times)),
                    "last_ms": {"upload": sol.ms_upload, "solve": sol.ms_solve, "download": sol.ms_download},
                    "trace_sha256": trace_digest(sol.trace)}
        plain, cached = timed_calls(False), timed_calls(True)
        h2d = 8 * (m * (n - m) + m + n)         # dense columns + b + c (the slack block is verified on the host, not copied)
        d2h = 8 * m + 4 * m + 8 * P + 64        # x_b, b_ixs, trace, result block
        e2e = {**plain, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "pivots_per_step": P,
               "note": "b200lp_solve_f64 per step with pinned host buffers, memory cache OFF (default): cudaMalloc of all "
                       "device state, H2D of the LP, the pivots, D2H of x_b / b_ixs / trace and cudaFree inside the timed region; "
                       "value = pivots / total time (mean step); cudaFree of 16 GB takes 9 ms or ~500 ms from call to call "
                       "(B200LP_TIMING=1), see ms_per_step_each / value_at_median_step"}
        e2e_cached = {**cached, "note": "same call with b200lp_set_memory_cache(1): device buffers survive between calls"}
        del A_np, A_pin

    peak, peak_src = measured_peak_gbs()
    bpp = bytes_per_pivot(m, n)
    achieved = bpp * pivots_timed / (total_ms * 1e-3) / 1e9
    traffic, traffic_src = profiled_traffic(args.workload, P)
    out = {
        "metric": "pivots/s, dense revised simplex (fp64)", "value": value, "unit": "pivots/s",
        "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_ms / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_for(args.workload, m, n, P),
        "engine": {"grid_ctas": grid, "parallelism": "1 GPU, persistent cooperative kernel"},
        "device_loop": {"value": value, "unit": "pivots/s", "note": "CUDA events around the pivot loop only (= value)"},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src, "bytes_per_pivot": bpp,
                     "bytes_per_launch": bpp * P, "kernel": "simplex_persistent<double>"},
        "gpu_launches": int(launches), "clocks": clk.summary(), "e2e": e2e, "e2e_cached": e2e_cached, **parity,
        "status_after": status_after, "pivots_timed": int(pivots_timed), "engine_event_ms": internal_ms,
    }
    return out


def cpu_baseline(wl, budget_s=20.0):
    """CPU oracle (port of the reference loop) on the host cores, bounded sample of the same LP."""
    import oracle
    m, n = wl["m"], wl["n"]
    A, b, c = oracle.gen_dense(m, n, SEED)
    k, done, t_used = 2, 0, 0.0
    while True:
        t0 = time.perf_counter()
        s = oracle.solve(A, b, c, eps=EPS, max_iter=k, trace_cap=1)
        dt = time.perf_counter() - t0
        done, t_used = s.pivots, dt
        if dt > budget_s / 3 or s.status != oracle.MAX_ITER or k >= 1 << 16:
            break
        k *= 4
    return {"value": done / t_used, "unit": "pivots/s", "cores": oracle.num_threads(), "kind": "port",
            "sample": f"first {done} pivots of the same LP (m={m}, n={n}), {t_used:.1f} s, OpenMP over all host threads"}


# ---------------------------------------------------------------- reference arm

def _pinned_lp(m, n):
    """Host buffers for the reference arm: pinned like the reference's own main() allocates them (cudaMallocHost,
    v4:408-414) when torch + CUDA are there, pageable numpy otherwise.  Returns (A col-major m x n, b, c, pinned?)."""
    import oracle
    try:
        import torch
        if not torch.cuda.is_available():
            raise RuntimeError("no CUDA")
        A_pin = torch.empty((n, m), dtype=torch.float64, pin_memory=True)
        b_pin = torch.empty(m, dtype=torch.float64, pin_memory=True)
        c_pin = torch.empty(n, dtype=torch.float64, pin_memory=True)
        oracle.gen_dense_into(A_pin.data_ptr(), b_pin.data_ptr(), c_pin.data_ptr(), m, n, SEED)
        return A_pin.numpy().T, b_pin.numpy(), c_pin.numpy(), True, (A_pin, b_pin, c_pin)
    except Exception:
        A, b, c = oracle.gen_dense(m, n, SEED)
        return A, b, c, False, None


def reference_workload(args, name, wl, P):
    """One workload on the reference's own v4 CUDA solve() (or the CPU port): per step one call from the slack basis
    with host buffers in / out, like main() calls it (v4:423)."""
    import oracle
    m, n = wl["m"], wl["n"]
    use_v4 = oracle.ref_available(np.float64) and not args.ref_cpu
    if use_v4:
        try:
            import torch
            use_v4 = torch.cuda.is_available()
        except Exception:
            use_v4 = False
    times, piv, loop_s, r = [], 0, 0.0, None
    if use_v4:
        A, b, c, pinned, keep = _pinned_lp(m, n)
        for s in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            r = oracle.ref_solve(A, b, c, eps=EPS, max_iter=P, trace_cap=P, always_readback=True)
            dt = time.perf_counter() - t0
            if s >= args.warmup:
                times.append(dt)
                piv += r.pivots
                loop_s += r.secs_loop
        kind, cores = "reference-gpu", 1
        sample = (f"reference v4 CUDA solve() (oracle/_ref/libv4ref_f64.so: fp64 retarget + init-grid/length/pointer-mode "
                  f"fixes, make_ref.sh P1-P8) on the B200, {P} iterations per step from the slack basis, "
                  f"{'pinned' if pinned else 'pageable'} host buffers in/out, cudaMalloc/cudaFree per call (v4:245-264, 370-377); "
                  f"1 host thread drives the GPU")
        extra = {"device_loop": {"value": piv / loop_s if loop_s > 0 else None, "unit": "pivots/s",
                                 "note": "host clock from after the init kernels (v4:283) to before the frees (v4:370), "
                                         "i.e. the loop plus the final read-back"},
                 "runs_on": "B200 (cuBLAS + CUB)", "host_buffers": "pinned" if pinned else "pageable"}
        del keep
    else:
        A, b, c = oracle.gen_dense(m, n, SEED)
        P = min(P, args.ref_pivots or 8)
        for s in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            r = oracle.solve(A, b, c, eps=EPS, max_iter=P, trace_cap=P)
            dt = time.perf_counter() - t0
            if s >= args.warmup:
                times.append(dt)
                piv += r.pivots
        kind, cores = "port", oracle.num_threads()
        sample = f"CPU oracle port, {P} iterations per step from the slack basis, {cores} OpenMP threads"
        extra = {"device_loop": None, "runs_on": "host CPU", "host_buffers": "pageable"}
    value = piv / sum(times)
    trace = np.stack([r.trace_p, r.trace_q], axis=1) if len(r.trace_p) else np.zeros((0, 2), np.int32)
    return {"value": value, "unit": "pivots/s", "ms_per_step": 1e3 * sum(times) / len(times),
            "ms_per_step_each": [round(1e3 * t, 1) for t in times],
            "value_at_median_step": (piv / len(times)) / float(np.median(times)),
            "config": config_for(name, m, n, P),
            "cpu_baseline": {"value": value, "unit": "pivots/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": "pivots/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            **parity_fields(name, P, trace, r.z), **extra}


def run_reference(args, wl):
    """The reference's own v4 CUDA solver on the same LP (rank 0 only); falls back to the CPU port."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return None
    P = args.pivots or wl["pivots"]
    main_ = reference_workload(args, args.workload, wl, P)
    out = {"impl": "reference", "metric": "pivots/s, dense revised simplex (fp64)", "value": main_["value"],
           "unit": "pivots/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": main_["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
           "dtype": "f64", "data": "synthetic"}
    out.update({k: v for k, v in main_.items() if k not in ("value", "unit", "ms_per_step")})
    extra = {}
    if args.gpus == 1:
        for name in [x for x in args.extras.split(",") if x and x != args.workload]:
            r = reference_workload(args, name, WORKLOADS[name], WORKLOADS[name]["pivots"])
            extra[name] = {k: r[k] for k in ("value", "unit", "ms_per_step", "config", "device_loop", "trace_sha256",
                                             "z_after_window", "trace_matches_golden") if k in r}
    if extra:
        out["extra"] = extra
    return out


# ---------------------------------------------------------------- CPU baselines of the smaller named configs (SURVEY 8(d3))

def cpu_extras(budget_s=20.0):
    """Rank 0, N=1 only: the CPU port on C2 (whole solve) and on a window of C3, and HiGHS dual simplex
    (scipy `highs-ds`, 1 thread — the stand-in for solver_glpk.cpp's glp_simplex, GLPK being absent) time-to-optimal on C2."""
    import oracle
    out = {}
    m, n = WORKLOADS["C2"]["m"], WORKLOADS["C2"]["n"]
    A, b, c = oracle.gen_dense(m, n, SEED)
    t0 = time.perf_counter()
    s = oracle.solve(A, b, c, eps=EPS, max_iter=1 << 30, trace_cap=1)
    dt = time.perf_counter() - t0
    out["C2_cpu_port_to_optimal"] = {"seconds": dt, "pivots": int(s.pivots), "pivots_per_s": s.pivots / dt, "z": s.z,
                                     "status": int(s.status), "cores": oracle.num_threads(), "kind": "port"}
    try:
        from scipy.optimize import linprog
        t0 = time.perf_counter()
        r = linprog(-c[:n - m], A_ub=A[:, :n - m], b_ub=b, method="highs-ds")
        dt = time.perf_counter() - t0
        out["C2_highs_ds_to_optimal"] = {"seconds": dt, "iterations": int(r.nit), "z": float(-r.fun), "status": int(r.status),
                                         "cores": 1, "rel_diff_vs_port": abs(-r.fun - s.z) / abs(s.z),
                                         "note": "scipy.optimize.linprog(method='highs-ds'); GLPK (solver_glpk.cpp:23) is not installed"}
    except Exception as exc:
        out["C2_highs_ds_to_optimal"] = {"unavailable": str(exc)}
    m, n = WORKLOADS["C3"]["m"], WORKLOADS["C3"]["n"]
    A, b, c = oracle.gen_dense(m, n, SEED)
    k, done, t_used = 8, 0, 0.0
    while True:
        t0 = time.perf_counter()
        s = oracle.solve(A, b, c, eps=EPS, max_iter=k, trace_cap=1)
        t_used, done = time.perf_counter() - t0, s.pivots
        if t_used > budget_s / 3 or s.status != oracle.MAX_ITER:
            break
        k *= 4
    out["C3_cpu_port_window"] = {"seconds": t_used, "pivots": int(done), "pivots_per_s": done / t_used,
                                 "cores": oracle.num_threads(), "kind": "port"}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="C4", choices=sorted(WORKLOADS))
    ap.add_argument("--pivots", type=int, default=0, help="pivots per step (0 = workload default)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--extras", default="C2,C3", help="comma list of extra single-GPU workloads reported under 'extra' (both arms)")
    ap.add_argument("--tto", default="C2,C3", help="comma list of workloads solved to optimality (time-to-optimal), '' = none")
    ap.add_argument("--tto-se", default="C2,C3,C4", help="workloads solved to optimality with steepest-edge pricing "
                                                         "(options.pricing_rule = 1; a different pivot sequence, same optimum)")
    ap.add_argument("--no-km", action="store_true", help="skip the Klee-Minty 20 solve (config 5a) under 'extra'")
    ap.add_argument("--ref-cpu", action="store_true", help="reference arm: force the CPU port")
    ap.add_argument("--ref-pivots", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write x_b, b_ixs, y, the (p, q) trace and z of the last timed window "
                         "of --workload as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    wl = WORKLOADS[args.workload]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        out = run_reference(args, wl)
        if out is not None:
            print(json.dumps(out), flush=True)
        return

    if args.gpus > 1 or world > 1:
        from simplex_method_gpu_b200 import sharded_bench
        out = sharded_bench.run(args, wl, SEED, EPS)
    else:
        out = run_b200_single(args, wl)
        if not args.no_cpu:
            out["cpu_baseline"] = cpu_baseline(wl)
        extra = {}
        if not args.no_cpu:
            extra["cpu"] = cpu_extras()
        for name in [x for x in args.extras.split(",") if x and x != args.workload]:
            sub = argparse.Namespace(**vars(args))
            sub.workload, sub.pivots, sub.no_e2e, sub.dump_outputs = name, 0, True, None
            r = run_b200_single(sub, WORKLOADS[name])
            extra[name] = {k: r[k] for k in ("value", "unit", "ms_per_step", "roofline", "config", "device_loop", "clocks",
                                             "gpu_launches", "trace_sha256", "z_after_window", "trace_matches_golden") if k in r}
        tto, tto_se = {}, {}
        dev = int(os.environ.get("LOCAL_RANK", "0"))
        for name in [x for x in args.tto.split(",") if x]:
            tto[name] = time_to_optimal(name, WORKLOADS[name], dev)
        for name in [x for x in args.tto_se.split(",") if x]:
            tto_se[name] = time_to_optimal(name, WORKLOADS[name], dev, rule=1)
        if not args.no_km:
            extra["klee_minty_20"] = klee_minty_20(dev)
        if tto:
            extra["time_to_optimal"] = tto
        if tto_se:
            extra["time_to_optimal_steepest_edge"] = tto_se
        if extra:
            out["extra"] = extra
    if rank == 0 and out is not None:
        print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()

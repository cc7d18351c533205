"""bench.py's N>1 arm: the sharded engine under torchrun, one rank per GPU."""
from __future__ import annotations

import json
import os
import time

import numpy as np


def run(args, wl, seed, eps):
    import torch
    import torch.distributed as dist

    from .sharded import ShardedEngine, ShardPlan
    from .solver import lpgen_dense_into

    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", str(rank)))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    m, n, P = wl["m"], wl["n"], args.pivots or wl["pivots"]
    plan = ShardPlan(m, n, world, 8)

    eng = ShardedEngine(m, n, np.float64, rank=rank, world=world, device=local, eps=eps, max_iter=1 << 40)
    eng.generate_dense(seed)
    eng.connect()
    stream = torch.cuda.ExternalStream(eng.stream, device=local)
    dist.barrier()

    def window():
        eng.reset()
        dist.barrier()
        torch.cuda.synchronize()
        a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = eng.run(0)["kernel_launches"]
        dist.barrier()
        a.record(stream)
        eng.run_async(P)
        b_.record(stream)
        r = eng.wait()
        torch.cuda.synchronize()
        return a.elapsed_time(b_), r, r["kernel_launches"] - l0

    ms, piv, launches = [], 0, 0
    from bench import ClockSampler          # same sampler as the single-GPU arm
    with ClockSampler(local) as clk:
        for _ in range(args.warmup):
            window()
        clk.mark_start()
        for _ in range(args.steps):
            t, r, l = window()
            ms.append(t)
            piv += r["pivots"]
            launches += l
        clk.mark_end()
    t_ms = torch.tensor(ms, dtype=torch.float64, device="cuda")
    dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)                 # device time, max over ranks
    total_ms = float(t_ms.sum().item())
    value = piv / (total_ms * 1e-3)
    x_b, b_ixs, y = eng.download()
    trace = eng.trace(P)
    if args.dump_outputs and rank == 0:     # the full x_b, b_ixs, y and trace, as the certificate below reads them
        from bench import dump_outputs
        dump_outputs(args.dump_outputs, {"x_b": x_b, "b_ixs": b_ixs, "y": y, "trace": trace, "z": [r["z"]]})
    digest = torch.tensor([float(r["pivots"]), float(r["z"]), float(np.asarray(b_ixs, np.float64).sum())],
                          dtype=torch.float64, device="cuda")
    lo, hi = digest.clone(), digest.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    replicas_agree = bool(torch.equal(lo, hi))

    # ---- end to end: every rank uploads its own column block from pinned host memory
    e2e = None
    if not args.no_e2e:
        c0, c1 = plan.cols(rank)
        A_pin = torch.empty((max(c1 - c0, 1), m), dtype=torch.float64, pin_memory=True)
        b_pin = torch.empty(m, dtype=torch.float64, pin_memory=True)
        c_pin = torch.empty(n, dtype=torch.float64, pin_memory=True)
        lpgen_dense_into(A_pin.data_ptr(), b_pin.data_ptr(), c_pin.data_ptr(), m, n, c0, c1 - c0, seed)
        A_cols = A_pin.numpy()[:c1 - c0].T
        times, piv2 = [], 0
        for s in range(args.warmup + args.steps):
            dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            eng.upload_columns(A_cols, b_pin.numpy(), c_pin.numpy())
            r2 = eng.run(P)
            xb2, ix2, _ = eng.download()
            torch.cuda.synchronize()
            dt = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            if s >= args.warmup:
                times.append(float(dt.item()))
                piv2 += r2["pivots"]
        e2e = {"value": piv2 / sum(times), "unit": "pivots/s",
               "h2d_bytes_per_step": 8 * (m * (n - m) + world * (m + n)), "d2h_bytes_per_step": world * (12 * m + 64),
               "ms_per_step": 1e3 * sum(times) / len(times), "pivots_per_step": P,
               "note": "each rank uploads its own column block of A (and b, c) from pinned host memory through "
                       "b200lp_upload_columns, runs the window and reads x_b / b_ixs back; device buffers are kept "
                       "between steps (handle API) — compare with the single-GPU arm's e2e_cached"}

    # ---- time to optimal with steepest-edge pricing on all ranks (options.pricing_rule = 1; same optimum, far fewer pivots)
    tto_se = None
    if getattr(args, "tto_se", "") and args.workload in args.tto_se.split(","):
        eng.close()
        eng = ShardedEngine(m, n, np.float64, rank=rank, world=world, device=local, eps=eps, max_iter=1 << 40, pricing_rule=1)
        eng.generate_dense(seed)
        eng.connect()
        dist.barrier()
        eng.run(4)
        eng.reset()
        dist.barrier()
        t0 = time.perf_counter()
        rs = eng.run(1 << 40)
        wall = time.perf_counter() - t0
        tms = torch.tensor([rs["ms_solve"]], dtype=torch.float64, device="cuda")
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        xs, ixs, ys = eng.download()
        tto_se = {"workload": f"{args.workload}: dense LP m={m} n={n}, seed {seed}, slack basis to optimum on {world} GPUs",
                  "pricing_rule": "steepest edge (Goldfarb-Reid recurrence)", "status": int(rs["status"]),
                  "pivots": int(rs["pivots"]), "iterations": int(rs["iterations"]), "z": rs["z"],
                  "seconds": float(tms.item()) * 1e-3, "wall_seconds": wall,
                  "pivots_per_s": rs["pivots"] / (float(tms.item()) * 1e-3)}
        if rank == 0:
            from bench import optimality_certificate
            tto_se["certificate"] = optimality_certificate(m, n, xs, ixs, ys, rs["z"])
        dist.barrier()

    from bench import bytes_per_pivot, config_for, measured_peak_gbs, parity_fields
    # every rank holds the replicated trace: all of them must carry the digest rank 0 prints
    sha_bytes = torch.tensor(list(bytes.fromhex(parity_fields(args.workload, P, trace, r["z"])["trace_sha256"])),
                             dtype=torch.int32, device="cuda")
    lo_s, hi_s = sha_bytes.clone(), sha_bytes.clone()
    dist.all_reduce(lo_s, op=dist.ReduceOp.MIN)
    dist.all_reduce(hi_s, op=dist.ReduceOp.MAX)
    replicas_agree = replicas_agree and bool(torch.equal(lo_s, hi_s))
    peak, peak_src = measured_peak_gbs()
    bpp = bytes_per_pivot(m, n)
    achieved = bpp * piv / (total_ms * 1e-3) / 1e9
    out = {
        "metric": "pivots/s, dense revised simplex (fp64)", "value": value, "unit": "pivots/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_ms / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_for(args.workload, m, n, P),
        "engine": {"grid_ctas": eng.grid_ctas,
                   "parallelism": f"{world} GPUs: B^-1 row-sharded, A column-sharded, peer-store exchanges (no NCCL on the data path)",
                   "l2": "per-GPU working set larger than L2" if bpp / world > 2 * 126e6 else "per-GPU working set near/below L2 size"},
        "device_loop": {"value": value, "unit": "pivots/s", "note": "CUDA events around the pivot loop only, max over ranks (= value)"},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak * world, "unit": "GB/s",
                     "frac": achieved / (peak * world), "traffic": None, "peak_source": peak_src + f" x {world} GPUs",
                     "bytes_per_pivot": bpp, "kernel": "simplex_persistent_sharded<double>"},
        "gpu_launches": int(launches), "clocks": clk.summary(), "e2e": e2e,
        "replicas_agree": replicas_agree, "pivots_timed": int(piv), **parity_fields(args.workload, P, trace, r["z"]),
        "exchange_bytes_per_pivot_per_rank": plan.exchange_bytes_per_pivot(),
    }
    if tto_se:
        out["extra"] = {"time_to_optimal_steepest_edge": {args.workload: tto_se}}
    eng.close()
    dist.barrier()
    dist.destroy_process_group()
    return out

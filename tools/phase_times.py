"""Dev tool (GPU box): per-phase time breakdown INSIDE the persistent kernel, from the %globaltimer
stamps CTA 0 records at every phase boundary (options.profile).  Single GPU:

    python tools/phase_times.py --lp 8192x16384 --pivots 300

Sharded (one rank per GPU):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 \
        --master-port 29531 tools/phase_times.py --lp 32768x65536 --pivots 64
"""
import argparse
import json
import os
import sys

import ctypes as C

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import simplex_method_gpu_b200 as lp  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--lp", default="8192x16384", help="MxN (not --m/--n: torchrun's argparse would grab them)")
ap.add_argument("--pivots", type=int, default=300)
ap.add_argument("--skip", type=int, default=20, help="leading pivots left out of the averages")
ap.add_argument("--grid", type=int, default=0)
ap.add_argument("--shape", type=int, default=0, help="update+FTRAN tile shape (warps along columns), 0 = auto")
ap.add_argument("--price-cols", type=int, default=0)
ap.add_argument("--l2", type=int, default=-1, help="l2_persist_mb: -1 off, 0 max, else MiB")
ap.add_argument("--price-mode", type=int, default=0, help="0 auto, 1 TMA ring, 2 register-staged")
ap.add_argument("--group-rows", type=int, default=0, help="ratio_group_rows (0 = auto)")
ap.add_argument("--tail", type=int, default=0, help="price_tail: 0 auto, -1 none, else columns")
ap.add_argument("--fuse", type=int, default=0, help="fuse_book2: 0 auto, -1 off")
ap.add_argument("--fuse-ratio", type=int, default=0, help="fuse_ratio: 0 auto, -1 off")
ap.add_argument("--rule", type=int, default=0, help="pricing_rule: 0 Dantzig, 1 steepest edge")
ap.add_argument("--binv-sparse", type=int, default=0, help="binv_sparse: 0 auto, -1 off (stream all of B^-1), else K*")
ap.add_argument("--resident", type=int, default=0, help="1: label the stamps of the shared-memory-resident kernel (mid-size LPs, auto configuration)")
ap.add_argument("--out", default="")
a = ap.parse_args()
a.m, a.n = (int(x) for x in a.lp.lower().split("x"))

world = int(os.environ.get("WORLD_SIZE", "1"))
rank = int(os.environ.get("RANK", "0"))
names = json.loads(lp.capi.lib().b200lp_profile_names().decode())

if world > 1:
    import torch
    import torch.distributed as dist
    from simplex_method_gpu_b200.sharded import ShardedEngine
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    e = ShardedEngine(a.m, a.n, np.float64, rank=rank, world=world, device=local, eps=1e-9, max_iter=1 << 30,
                      profile=a.pivots, grid_ctas=a.grid, tile_shape=a.shape, price_cols=a.price_cols, l2_persist_mb=a.l2, price_mode=a.price_mode,
                      ratio_group_rows=a.group_rows, price_tail=a.tail, fuse_book2=a.fuse, fuse_ratio=a.fuse_ratio, pricing_rule=a.rule)
    e.generate_dense(1)
    e.connect()
    dist.barrier()
    names = names["sharded"]
else:
    e = lp.Engine(a.m, a.n, np.float64, eps=1e-9, max_iter=1 << 30, profile=a.pivots, grid_ctas=a.grid, tile_shape=a.shape, price_cols=a.price_cols, l2_persist_mb=a.l2, price_mode=a.price_mode,
                      ratio_group_rows=a.group_rows, price_tail=a.tail, fuse_book2=a.fuse, fuse_ratio=a.fuse_ratio, pricing_rule=a.rule,
                      binv_sparse=a.binv_sparse)
    e.generate_dense(1)
    names = names["resident"] if a.resident else names["single"]

e.run(8)                                  # warm-up launch
r0 = e.run(0)
r = e.run(a.pivots)
st = e.profile().astype(np.int64)         # (iterations, stamps)
piv = r["pivots"] - r0["pivots"]
k = len(names)
st = st[a.skip:, :k]
st = st[st[:, 0] > 0]
for j in range(1, k):                     # a point the loop did not pass (fused book2): zero-length interval
    st[:, j] = np.where(st[:, j] == 0, st[:, j - 1], st[:, j])
# stamp j of iteration i+1 closes the last interval of iteration i
nxt = np.roll(st[:, 0], -1)
full = np.concatenate([st, nxt[:, None]], axis=1)[:-1]
d = np.diff(full, axis=1) / 1e3           # us
tot = d.sum(axis=1)
lines = [f"rank {rank}/{world}  m={a.m} n={a.n} grid={e.grid_ctas}: {piv} pivots in {r['ms_solve']:.2f} ms "
         f"({r['ms_solve'] / max(piv, 1) * 1e3:.1f} us/pivot by events); {len(d)} iterations averaged, "
         f"{tot.mean():.1f} us/iteration by stamps"]
for j in range(k):
    lines.append(f"  {names[j]:<44s} {d[:, j].mean():8.2f} us  (min {d[:, j].min():7.2f}, max {d[:, j].max():7.2f})  "
                 f"{100 * d[:, j].mean() / tot.mean():5.1f}%")
text = "\n".join(lines)
if world > 1:
    import torch.distributed as dist
    gathered = [None] * world
    dist.all_gather_object(gathered, text)
    text = "\n".join(gathered)
if rank == 0:
    print(text, flush=True)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")
e.close()
if world > 1:
    dist.barrier()
    dist.destroy_process_group()

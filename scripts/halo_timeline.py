"""Multi-rank apply: single-launch (fused) path vs the NCCL exchange on the SAME box and operator, plus a %globaltimer
timeline of the fused kernel's roles on every rank. Launch with torchrun (one process per GPU):
  python -m torch.distributed.run --nproc-per-node N --master-addr 127.0.0.1 scripts/halo_timeline.py [--size 256] [--nvec 1]"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
import torch.distributed as dist

import bench
import maxwell_b200 as mx

ap = argparse.ArgumentParser()
ap.add_argument("--size", type=int, default=256)
ap.add_argument("--workload", default="pillbox")
ap.add_argument("--nvecs", default="1,4")
ap.add_argument("--reps", type=int, default=200)
args = ap.parse_args()
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
local_rank = int(os.environ.get("LOCAL_RANK", rank))
dist.init_process_group("gloo", rank=rank, world_size=world)
sizes = [args.size]
if rank == 0:
    bench.ensure_generated(args.workload, args.size, sizes, False, 2)
dist.barrier()
store = bench.OpStore(args.workload, args.size)
ctx = mx.Context(local_rank)
ids = [mx.Context.unique_id() if rank == 0 else None]
dist.broadcast_object_list(ids, src=0)
ctx.comm_init(rank, world, ids[0])
m = store.load("L%d.curlCurl" % args.size)
rg = np.asarray(m["rg"])
n_global = int(m["n_global"][0])
cuts = bench.slab_ranges(rg, n_global, world, args.size)
r0, r1 = cuts[rank], cuts[rank + 1]
bmap = mx.MxMap(ctx, n_global, np.ascontiguousarray(rg[r0:r1]))
ops = {}
for name, env in (("fused", {}), ("nccl", {"MXG_HALO": "nccl"})):
    os.environ.pop("MXG_HALO", None)
    os.environ.update(env)
    ops[name] = bench.upload_block(mx, m, bmap, bmap, r0, r1)
out = {"world": world, "rows_rank0": int(r1 - r0)}
for nv in [int(v) for v in args.nvecs.split(",")]:
    x = mx.MxMultiVector(bmap, nv)
    y = mx.MxMultiVector(bmap, nv)
    x.random(12345)
    ref = None
    for name, A in ops.items():
        for _ in range(10):
            A.apply(x, y)
        ctx.sync()
        dist.barrier()
        ctx.event_record(0)
        for _ in range(args.reps):
            A.apply(x, y)
        ctx.event_record(1)
        ms = ctx.event_elapsed_ms(0, 1) / args.reps
        ctx.sync()
        t = torch.tensor([ms], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        yh = y.to_host()
        if ref is None:
            ref = yh
        same = bool(np.array_equal(ref, yh))
        out["%s_nvec%d" % (name, nv)] = {"ms": round(float(t[0]), 4), "same_as_first": same}
    # timeline of the fused kernel (each rank its own clock origin)
    A = ops["fused"]
    tl = []
    for _ in range(3):
        dist.barrier()
        tl.append(A.trace_apply(x, y))
    mine = {k: [round(v[0] / 1e3, 1), round(v[1] / 1e3, 1)] for k, v in tl[-1].items()}
    allt = [None] * world
    dist.all_gather_object(allt, mine)
    out["timeline_us_nvec%d" % nv] = allt
    del x, y
if rank == 0:
    print(json.dumps(out))
dist.barrier()
dist.destroy_process_group()

"""Per-rank cost of the slab-partitioned device assembly (include/mxasm.h: mxg_sim_op_rows and the transfer rows) on one
GPU: wall time and peak assembly bytes (mxg_asm_memory) of

  - the replicated build: pillbox-256, the whole hierarchy of the eigensolve (bench.py's level list for one rank), as
    EigenProblem builds it (operators, transfers, layouts);
  - the slab builds: pillbox-256, every virtual rank of worlds 2, 4 and 8 one after another in this process, the
    operators and transfers of that rank's rows (bench.py's level list for that world);
  - one middle slab (rank 3 of 8) of pillbox-512 and of the 512-cell crab cavity (cell_res = 127, 318 x 318 x 512).

The fractions and DOF maps stay global on every rank; their resident bytes are reported separately ("sims_bytes"). The
slab builds measure the assembly only: the layouts of a slab need the other ranks' halo plan (run under torchrun).
The card's name and power limit are read in the same run. Usage: python scripts/slab_assembly_bench.py [--out FILE]
[--skip-512]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import maxwell_b200 as mx  # noqa: E402
from maxwell_b200 import assembly as asm  # noqa: E402
from maxwell_b200.partition import slab_cuts  # noqa: E402

GB = 1e9


def level_sizes(size, world, workload):
    """bench.py's level list (coarsest level 8^3 on 1-2 ranks, 16^3 from 4 ranks on; crab cavity: one level)."""
    if workload == "crabcav":
        return [size]
    sizes = [size]
    floor = 8 if world <= 2 else 16
    while sizes[-1] % 2 == 0 and sizes[-1] // 2 >= floor and len(sizes) < 6:
        sizes.append(sizes[-1] // 2)
    return sizes


def card():
    try:
        out = subprocess.check_output(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"], text=True)
        name, limit = [s.strip() for s in out.strip().splitlines()[0].split(",")]
        return {"name": name, "power_limit": limit}
    except Exception as e:           # the numbers are still reported; say why the card is unknown
        return {"name": "unknown (%s)" % e, "power_limit": "unknown"}


def ranges(sims, sizes, rank, world):
    rng = {}
    for l, s in enumerate(sims):
        for f in ("bfield", "psifield"):
            if world == 1:
                rng[l, f] = (0, s.map_size(f)[0])
            else:
                c = slab_cuts(s.map(f), s.num_global(f), sizes[l] + 1, world)
                rng[l, f] = (c[rank], c[rank + 1])
    return rng


def assemble_rows(sims, rng, cx=False):
    """The matrices EigenProblem assembles for these rows, each released once built (as EigenProblem does after its layout)."""
    nnz = 0
    for l, s in enumerate(sims):
        nnz += s.op("vecLapl", cx, rows=rng[l, "bfield"]).nnz
        nnz += s.op("scaLapl", cx, rows=rng[l, "psifield"]).nnz
    for l in range(len(sims) - 1):
        for f in ("bfield", "psifield"):
            nnz += sims[l].interpolator_from(sims[l + 1], f, cx, rows=rng[l, f]).nnz
            nnz += sims[l].interpolator_transpose(sims[l + 1], f, cx, rows=rng[l + 1, f]).scale(0.125).nnz
    s0 = sims[0]
    nnz += s0.op("divB", cx, rows=rng[0, "psifield"]).nnz
    for name in ("gradPsi", "curlCurl", "dmA"):
        nnz += s0.op(name, cx, rows=rng[0, "bfield"]).nnz
    return nnz


def measure(ctx, fn):
    ctx.sync()
    base, _ = asm.asm_memory(ctx, reset_peak=True)
    t = time.time()
    r = fn()
    ctx.sync()
    dt = time.time() - t
    _, peak = asm.asm_memory(ctx)
    return r, round(dt, 4), peak - base


def sims_for(ctx, workload, sizes):
    ctx.sync()
    t = time.time()
    sims = [asm.example_sim(ctx, workload, n) for n in sizes]
    ctx.sync()
    return sims, round(time.time() - t, 4), asm.asm_memory(ctx)[0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--skip-512", action="store_true")
    args = ap.parse_args()
    ctx = mx.Context(0)
    res = {"gpu": card(), "units": "seconds, bytes above the post-set-up baseline (peak_bytes), resident bytes (sims_bytes)"}
    print(json.dumps({"gpu": res["gpu"]}), flush=True)
    warm = asm.example_sim(ctx, "pillbox", 16)        # kernels loaded once
    assemble_rows([warm], {(0, "bfield"): (0, warm.map_size("bfield")[0]), (0, "psifield"): (0, warm.map_size("psifield")[0])})
    del warm

    sizes = level_sizes(256, 1, "pillbox")
    sims, t_setup, sims_bytes = sims_for(ctx, "pillbox", sizes)
    ep, t_ep, peak_ep = measure(ctx, lambda: asm.EigenProblem(ctx, sims))
    del ep
    nnz, t_rows, peak_rows = measure(ctx, lambda: assemble_rows(sims, ranges(sims, sizes, 0, 1)))
    rep = {"levels": sizes, "sims_setup_s": t_setup, "sims_bytes": sims_bytes, "eigenproblem_s": t_ep, "eigenproblem_peak_bytes": peak_ep,
           "assembly_s": t_rows, "assembly_peak_bytes": peak_rows, "nnz": nnz}
    res["pillbox256_replicated"] = rep
    print(json.dumps({"pillbox256_replicated": rep}), flush=True)
    del sims

    res["pillbox256_slabs"] = {}
    for world in (2, 4, 8):
        sizes = level_sizes(256, world, "pillbox")
        sims, t_setup, sims_bytes = sims_for(ctx, "pillbox", sizes)
        per = []
        for rank in range(world):
            nnz, t, peak = measure(ctx, lambda: assemble_rows(sims, ranges(sims, sizes, rank, world)))
            per.append({"rank": rank, "assembly_s": t, "assembly_peak_bytes": peak, "nnz": nnz})
        w = {"levels": sizes, "sims_setup_s": t_setup, "sims_bytes": sims_bytes, "ranks": per,
             "max_assembly_s": max(p["assembly_s"] for p in per), "max_assembly_peak_bytes": max(p["assembly_peak_bytes"] for p in per)}
        res["pillbox256_slabs"][str(world)] = w
        print(json.dumps({"pillbox256_world%d" % world: w}), flush=True)
        del sims

    if not args.skip_512:
        for workload in ("pillbox", "crabcav"):
            sizes = level_sizes(512, 8, workload)
            sims, t_setup, sims_bytes = sims_for(ctx, workload, sizes)
            nnz, t, peak = measure(ctx, lambda: assemble_rows(sims, ranges(sims, sizes, 3, 8)))
            grid = list(sims[0].n)
            r = {"grid": grid, "levels": sizes, "rank": 3, "world": 8, "sims_setup_s": t_setup, "sims_bytes": sims_bytes,
                 "assembly_s": t, "assembly_peak_bytes": peak, "nnz": nnz}
            res["%s512_middle_slab" % workload] = r
            print(json.dumps({"%s512_middle_slab" % workload: r}), flush=True)
            del sims

    print("card: %s, power limit %s" % (res["gpu"]["name"], res["gpu"]["power_limit"]))
    rep = res["pillbox256_replicated"]
    print("%-34s %9s %12s %12s" % ("build", "time [s]", "peak [GB]", "sims [GB]"))
    print("%-34s %9.3f %12.2f %12.2f" % ("pillbox-256 EigenProblem, 1 rank", rep["eigenproblem_s"], rep["eigenproblem_peak_bytes"] / GB, rep["sims_bytes"] / GB))
    print("%-34s %9.3f %12.2f %12.2f" % ("pillbox-256 assembly, 1 rank", rep["assembly_s"], rep["assembly_peak_bytes"] / GB, rep["sims_bytes"] / GB))
    for world, w in res["pillbox256_slabs"].items():
        print("%-34s %9.3f %12.2f %12.2f" % ("pillbox-256 slab, world %s (max)" % world, w["max_assembly_s"], w["max_assembly_peak_bytes"] / GB,
                                             w["sims_bytes"] / GB))
    for workload in ("pillbox", "crabcav"):
        r = res.get("%s512_middle_slab" % workload)
        if r:
            print("%-34s %9.3f %12.2f %12.2f" % ("%s-512 rank 3 of 8" % workload, r["assembly_s"], r["assembly_peak_bytes"] / GB, r["sims_bytes"] / GB))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()

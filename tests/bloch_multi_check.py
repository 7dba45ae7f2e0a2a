"""Multi-GPU check of the Bloch transfers (DESIGN.md GMG-bloch), launched with torchrun by tests/test_gpu_multi_bloch.py (one
process per GPU). Every rank assembles its x-slab of a periodic-x Bloch problem with bloch_transfers: the slab rows of P and
R must apply like the oracle's global Bloch transfers, and the 2-level vector and scalar V-cycles must equal the float64
reference on the global operators to 1e-12 per column."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch.distributed as dist  # noqa: E402

import gmg_reference as G  # noqa: E402
import maxwell_b200 as mx  # noqa: E402
from maxwell_b200 import assembly as asm  # noqa: E402
from maxwell_b200.partition import slab_cuts  # noqa: E402
import bloch_oracle as BO  # noqa: E402
from oracle import oracle as orc  # noqa: E402
from slab_assembly_check import compare  # noqa: E402

PHI = (0.7, -0.4, 1.1)


def bloch_case(ctx, rank, world):
    sizes = [16, 8]
    sims = [asm.gpu_sim(ctx, n, origin=(0.0,) * 3, size=(1.0,) * 3, phase_shifts=PHI).setup() for n in sizes]
    osims = [orc.vacuum(n, phase_shifts=PHI) for n in sizes]

    def rows(l, f):
        c = slab_cuts(osims[l].map(f), osims[l].num_global(f), sizes[l] + 1, world)
        return c[rank], c[rank + 1]

    ep = asm.EigenProblem(ctx, sims, cuts=lambda l, f, gids, ng: rows(l, f), is_complex=True, bloch_transfers=True)
    for f, maps, P, R in (("bfield", ep.bmaps, ep.Pb, ep.Rb), ("psifield", ep.pmaps, ep.Pp, ep.Rp)):
        po = BO.interpolator(osims[1], osims[0], field=f, is_complex=True, bloch=True)
        compare(P[0], po, maps[0], maps[1], rows(0, f), "P " + f, is_complex=True, stats=False)
        compare(R[0], po.transpose(scale=0.125), maps[1], maps[0], rows(1, f), "R " + f, is_complex=True, stats=False)
    if rank == 0:
        print("case Bloch slab transfers ok on %d ranks" % world, flush=True)
    for name, field, ops, R, P, maps in (("vecLapl", "bfield", ep.vops, ep.Rb, ep.Pb, ep.bmaps),
                                         ("scaLapl", "psifield", ep.sops, ep.Rp, ep.Pp, ep.pmaps)):
        prec = mx.MxGeoMultigridPrec(ctx, ops, R, P, smoother_sweeps=2)
        oops = [s.op(name) for s in osims]
        gids = [op.maps()[0] for op in oops]
        Po = [BO.interpolator(osims[1], osims[0], field=field, is_complex=True, bloch=True)]
        Ro = [Po[0].transpose(scale=0.125)]
        ref = G.from_oracle(oops, Ro, Po, gids, lambda_max=[prec.info(l)["lambda_max"] for l in range(2)], smoother_sweeps=2)
        b = G.random_columns(41, gids[0], 2, True)
        c0, c1 = rows(0, field)
        bs = mx.MxMultiVector(maps[0], 2, True)
        bs.from_host(b[c0:c1])
        xs = bs.Clone(2)
        prec.ApplyInverse(bs, xs)
        err = G.column_errors(xs.to_host(), ref.apply(b)[c0:c1])
        assert np.all(err < 1e-12), (name, err)
    if rank == 0:
        print("case Bloch V-cycles equal the global reference on %d ranks" % world, flush=True)


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local_rank = int(os.environ.get("LOCAL_RANK", rank))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    ctx = mx.Context(local_rank)
    ids = [mx.Context.unique_id() if rank == 0 else None]
    dist.broadcast_object_list(ids, src=0)
    ctx.comm_init(rank, world, ids[0])
    bloch_case(ctx, rank, world)
    dist.barrier()
    print("RANK %d OK" % rank, flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()

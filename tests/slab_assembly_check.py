"""Multi-GPU check of the slab-partitioned assembly, launched with torchrun by tests/test_gpu_multi_slab.py (one process per
GPU). Every rank assembles only the rows of its x-slab (EigenProblem with cuts): the layouts must equal those the oracle's
rows of the same slab give, the applies must equal the oracle's global apply, and the projected eigensolve must return the
modes of the global pencil."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch.distributed as dist  # noqa: E402

import maxwell_b200 as mx  # noqa: E402
from maxwell_b200 import assembly as asm  # noqa: E402
from maxwell_b200.partition import local_block, slab_cuts  # noqa: E402
from multi_rank_check import _assert_matches_global  # noqa: E402
from oracle import oracle as orc  # noqa: E402


def slab_problem(ctx, rank, world, sims, sizes, is_complex=False):
    def cuts(l, f, gids, n_global):
        c = slab_cuts(gids, n_global, sizes[l] + 1, world)
        return c[rank], c[rank + 1]
    return asm.EigenProblem(ctx, sims, cuts=cuts, is_complex=is_complex)


def compare(A, oop, rmap, cmap, rcuts_rows, what, is_complex=False, stats=True):
    """A (device slab layout) against the oracle operator oop: same layout statistics as the oracle's slab rows, and an
    apply equal to the oracle's global apply."""
    rowptr, col, val = oop.arrays()
    rg, cg = oop.maps()
    r0, r1 = rcuts_rows
    if stats:
        lrp, lcol, lval = local_block(rowptr, cg[col], val, r0, r1)
        H = mx.MxCrsMatrix.from_csr(rmap, cmap, lrp, lcol, lval)
        assert A.stats() == H.stats(), (what, A.stats(), H.stats())
    x = mx.MxMultiVector(cmap, 2, is_complex)
    x.random(91)
    xg = np.empty((len(cg), 2), dtype=x.dtype)
    for j in range(2):
        xg[:, j] = mx.hash_uniform(91, cg, j, 0)
        if is_complex:
            xg[:, j] += 1j * mx.hash_uniform(91, cg, j, 1)
    y = mx.MxMultiVector(rmap, 2, is_complex)
    A.apply(x, y)
    _assert_matches_global(y.to_host(), oop.apply(xg)[r0:r1], is_complex, (what,))


def pillbox_case(ctx, rank, world):
    import scipy.sparse as sp
    import scipy.sparse.linalg as sla
    sizes = [24, 12]
    sims = [asm.example_sim(ctx, "pillbox", n) for n in sizes]
    osims = [orc.pillbox(n) for n in sizes]
    ep = slab_problem(ctx, rank, world, sims, sizes)

    def rows(l, f):
        gids = osims[l].map(f)
        c = slab_cuts(gids, osims[l].num_global(f), sizes[l] + 1, world)
        return c[rank], c[rank + 1]

    of = osims[0]
    compare(ep.curlCurl, of.op("curlCurl"), ep.bmaps[0], ep.bmaps[0], rows(0, "bfield"), "curlCurl")
    for l in range(2):
        compare(ep.vops[l], osims[l].op("vecLapl"), ep.bmaps[l], ep.bmaps[l], rows(l, "bfield"), "vecLapl L%d" % l)
        compare(ep.sops[l], osims[l].op("scaLapl"), ep.pmaps[l], ep.pmaps[l], rows(l, "psifield"), "scaLapl L%d" % l)
    compare(ep.divB, of.op("divB"), ep.pmaps[0], ep.bmaps[0], rows(0, "psifield"), "divB")
    compare(ep.gradPsi, of.op("gradPsi"), ep.bmaps[0], ep.pmaps[0], rows(0, "bfield"), "gradPsi")
    for f, maps, P, R in (("bfield", ep.bmaps, ep.Pb, ep.Rb), ("psifield", ep.pmaps, ep.Pp, ep.Rp)):
        po = orc.interpolator(osims[1], osims[0], field=f)
        compare(P[0], po, maps[0], maps[1], rows(0, f), "P " + f)
        compare(R[0], po.transpose(scale=0.125), maps[1], maps[0], rows(1, f), "R " + f)
    fa = of.fracs("bfield")
    b0, b1 = rows(0, "bfield")
    assert np.array_equal(ep.fracs, of.op("dmA").arrays()[2][b0:b1])
    if rank == 0:
        print("case slab layouts and applies ok on %d ranks" % world, flush=True)

    prec = mx.MxGeoMultigridPrec(ctx, ep.vops, ep.Rb, ep.Pb, smoother_sweeps=2)
    sprec = mx.MxGeoMultigridPrec(ctx, ep.sops, ep.Rp, ep.Pp, smoother_sweeps=2, remove_const_field=True)
    nev = 6
    s = mx.MxSolver(ctx, ep.vops[0], m_diag=ep.m_diag, prec=prec, nev=nev, block_size=10, tol=1e-9, max_iters=300,
                    projection={"divB": ep.divB, "gradPsi": ep.gradPsi, "scaLapl": ep.sops[0], "sca_prec": sprec})
    ev = s.solve()
    assert s.converged == nev, (s.converged, s.residuals)
    keep = np.where(fa > 0)[0]
    A = of.op("curlCurl").scipy()[keep][:, keep].tocsc()
    ref = np.sort(sla.eigsh(A, k=3 * nev, M=sp.diags(fa[keep]).tocsc(), sigma=60.0, which="LM", tol=1e-13, return_eigenvectors=False))
    ref = ref[ref > 1e-6 * ref.max()][:nev]
    np.testing.assert_allclose(ev, ref, rtol=1e-9)
    if rank == 0:
        print("case slab-assembled projected eigensolve ok on %d ranks" % world, flush=True)


def bloch_case(ctx, rank, world):
    """Periodic x with Bloch phases: rank 0's chains reach the top planes through the wrap."""
    n, phases = 12, (0.4, -1.3, 2.2)
    d = asm.gpu_sim(ctx, n, origin=(0.0,) * 3, size=(1.0,) * 3, phase_shifts=phases).setup()
    o = orc.vacuum(n, phase_shifts=phases)
    gids = o.map("bfield")
    assert np.array_equal(gids, d.map("bfield"))
    c = slab_cuts(gids, o.num_global("bfield"), n + 1, world)
    bmap = asm.make_map(d, "bfield", c[rank], c[rank + 1])
    A = asm.to_crs(d.op("curlCurl", True, rows=(c[rank], c[rank + 1])), bmap, bmap)
    compare(A, o.op("curlCurl"), bmap, bmap, (c[rank], c[rank + 1]), "bloch curlCurl", is_complex=True, stats=False)
    if rank == 0:
        print("case periodic Bloch slab curl-curl ok on %d ranks" % world, flush=True)


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local_rank = int(os.environ.get("LOCAL_RANK", rank))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    ctx = mx.Context(local_rank)
    ids = [mx.Context.unique_id() if rank == 0 else None]
    dist.broadcast_object_list(ids, src=0)
    ctx.comm_init(rank, world, ids[0])
    pillbox_case(ctx, rank, world)
    bloch_case(ctx, rank, world)
    dist.barrier()
    print("RANK %d OK" % rank, flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()

"""Multi-GPU parity script, launched with torchrun by tests/test_gpu_multi.py (one process per GPU).
Checks the NCCL halo exchange inside mxg_crs_apply and the all-reduced block reductions against the
oracle's global (single-process) results. P-invariance: x is generated from global ids, so every rank
count sees the same vector."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch.distributed as dist  # noqa: E402

import maxwell_b200 as mx  # noqa: E402
from maxwell_b200.partition import local_block, slab_cuts  # noqa: E402
from oracle import oracle as orc  # noqa: E402
import gmg_reference  # noqa: E402


def _assert_matches_global(got, ref, is_complex, what):
    """bit for bit for real operators, to 1e-14 (relative 2-norm) for complex ones"""
    if is_complex:
        err = np.linalg.norm(got - ref) / np.linalg.norm(ref)
        assert err < 1e-14, what + (err,)
    else:
        assert np.array_equal(got, ref), what + ("halo apply differs from the global apply",)


def _block(m, cuts, rank):
    rowptr, col, val = m.arrays()
    rg, cg = m.maps()
    return local_block(rowptr, cg[col], val, cuts[rank], cuts[rank + 1])


def solve_case(ctx, rank, world):
    """Multigrid (V-cycle and full multigrid) + the projected eigensolve on `world` ranks: every level operator, transfer and
    projection operator is slab-partitioned, the halo exchange runs inside every apply. The eigenvalues must equal scipy's on
    the global curl-curl pencil (gradient space deflated at 0) to 1e-9, i.e. be independent of the rank count."""
    import scipy.sparse as sp
    import scipy.sparse.linalg as sla
    sizes = [24, 12]
    sims = [orc.pillbox(n) for n in sizes]

    def part(sim, field, n):
        gids = sim.map(field)
        ng = sim.num_global(field)
        cuts = slab_cuts(gids, ng, n + 1, world)
        return gids, ng, cuts, mx.MxMap(ctx, ng, gids[cuts[rank]:cuts[rank + 1]])

    B = [part(s, "bfield", n) for s, n in zip(sims, sizes)]
    Ps = [part(s, "psifield", n) for s, n in zip(sims, sizes)]

    def up(mat, rowpart, colpart):
        lrp, lcol, lval = _block(mat, rowpart[2], rank)
        return mx.MxCrsMatrix.from_csr(rowpart[3], colpart[3], lrp, lcol, lval)

    vops = [up(s.op("vecLapl"), b, b) for s, b in zip(sims, B)]
    sops = [up(s.op("scaLapl"), p, p) for s, p in zip(sims, Ps)]
    pb = orc.interpolator(sims[1], sims[0])
    pp = orc.interpolator(sims[1], sims[0], field="psifield")
    Pb, Rb = [up(pb, B[0], B[1])], [up(pb.transpose(scale=0.125), B[1], B[0])]
    Pp, Rp = [up(pp, Ps[0], Ps[1])], [up(pp.transpose(scale=0.125), Ps[1], Ps[0])]
    D = up(sims[0].op("divB"), Ps[0], B[0])
    G = up(sims[0].op("gradPsi"), B[0], Ps[0])
    CC = up(sims[0].op("curlCurl"), B[0], B[0])
    fa = sims[0].fracs("bfield")
    cuts = B[0][2]
    md = mx.MxMultiVector(B[0][3], 1)
    md.from_host(fa[cuts[rank]:cuts[rank + 1]])

    def matches_reference(prec, parts, name, field, b, what, **kw):
        """This rank's slab of M^-1 b equals the matching rows of the float64 reference cycle on the global operators (run with
        the all-reduced lambda_max of the GPU, which is the restated power iteration's to rounding) to 1e-12 per column."""
        ops, R, P, gids = gmg_reference.oracle_hierarchy(orc, sims, name, field)
        lam = [prec.info(l)["lambda_max"] for l in range(len(sims))]
        ref = gmg_reference.from_oracle(ops, R, P, gids, lambda_max=lam, **kw)
        for l in range(len(sims)):
            want = gmg_reference.power_lambda_max(ref.A[l], ref.dinv[l], gids[l], l)
            assert abs(lam[l] - want) <= 1e-12 * want, what + ("lambda_max", l, lam[l], want)
        c0, c1 = parts[0][2][rank], parts[0][2][rank + 1]
        bs = mx.MxMultiVector(parts[0][3], b.shape[1])
        bs.from_host(b[c0:c1])
        xs = bs.Clone(b.shape[1])
        prec.ApplyInverse(bs, xs)
        err = gmg_reference.column_errors(xs.to_host(), ref.apply(b)[c0:c1])
        assert np.all(err < 1e-12), what + (err,)
        return bs, xs

    for fmg in (True, False):
        prec = mx.MxGeoMultigridPrec(ctx, vops, Rb, Pb, smoother_sweeps=2, full_multigrid=fmg)
        bg = gmg_reference.random_columns(21, B[0][0], 2, False) * (fa > 0)[:, None]
        b, x = matches_reference(prec, B, "vecLapl", "bfield", bg, ("multigrid on %d ranks" % world, fmg), full_multigrid=fmg)
        r = b.CloneCopy()
        vops[0].apply_axpby(-1.0, x, 1.0, r)
        red = (r.norm2() / b.norm2()).max()
        assert red < 0.8, ("multigrid on %d ranks" % world, fmg, red)
    sprec = mx.MxGeoMultigridPrec(ctx, sops, Rp, Pp, smoother_sweeps=2, remove_const_field=True)
    bg = gmg_reference.random_columns(23, Ps[0][0], 2, False)
    matches_reference(sprec, Ps, "scaLapl", "psifield", bg, ("scalar multigrid on %d ranks" % world,), remove_const_field=True)
    nev = 6
    s = mx.MxSolver(ctx, vops[0], m_diag=md, prec=prec, nev=nev, block_size=10, tol=1e-9, max_iters=300,
                    projection={"divB": D, "gradPsi": G, "scaLapl": sops[0], "sca_prec": sprec})
    ev = s.solve()
    assert s.converged == nev, (s.converged, s.residuals)
    keep = np.where(fa > 0)[0]
    A = sims[0].op("curlCurl").scipy()[keep][:, keep].tocsc()
    ref = np.sort(sla.eigsh(A, k=3 * nev, M=sp.diags(fa[keep]).tocsc(), sigma=60.0, which="LM", tol=1e-13, return_eigenvectors=False))
    ref = ref[ref > 1e-6 * ref.max()][:nev]
    np.testing.assert_allclose(ev, ref, rtol=1e-9)
    res, div = s.check(D, A=CC)
    assert np.all(res[:nev] < 1e-6) and np.all(div[:nev] < 1e-6), (res[:nev], div[:nev])
    if rank == 0:
        print("case multigrid + projected eigensolve ok on %d ranks" % world, flush=True)


def dense_case(ctx, rank, world):
    """Block products and reductions on ragged partitions: one rank owns no rows, or one owns fewer than 64 (a single tail
    chunk). The data are small integers and the scalars dyadic, so every partial sum is an integer below 2^53: the all-reduced
    Gram, dot, norm and mean and each rank's rows of the update must equal the global numpy result bit for bit, whatever
    the rank count."""
    n = 1 << 16                                       # a power of two: remove_const_field's 1/count is exact
    rng = np.random.default_rng(64)                   # the same global data on every rank
    Ag = rng.integers(-8, 9, size=(n, 72)).astype(np.float64)
    Xg = rng.integers(-8, 9, size=(n, 24)).astype(np.float64)
    Cg = rng.integers(-8, 9, size=(n, 5)) + 1j * rng.integers(-8, 9, size=(n, 5))
    B = rng.integers(-4, 5, size=(72, 24)).astype(np.float64)
    gids = np.arange(n, dtype=np.int64)

    def even(total, parts):
        return [total // parts + (1 if i < total % parts else 0) for i in range(parts)]

    for label, sizes in (("rank 0 owns no rows", [0] + even(n, world - 1)),
                         ("the last rank owns 37 rows", even(n - 37, world - 1) + [37])):
        cuts = np.concatenate([[0], np.cumsum(sizes)])
        r0, r1 = int(cuts[rank]), int(cuts[rank + 1])
        m = mx.MxMap(ctx, n, gids[r0:r1])
        A, X, Cx = mx.MxMultiVector(m, 72), mx.MxMultiVector(m, 24), mx.MxMultiVector(m, 5, True)
        A.from_host(Ag[r0:r1])
        X.from_host(Xg[r0:r1])
        Cx.from_host(Cg[r0:r1])
        what = (label, world)
        assert np.array_equal(X.MvTransMv(-0.5, A.CloneView(list(range(40)))), -0.5 * (Ag[:, :40].T @ Xg)), what + ("gram",)
        assert np.array_equal(X.MvTransMv(2.0, A), 2.0 * (Ag.T @ Xg)), what + ("gram, 72 columns",)
        assert np.array_equal(Cx.MvTransMv(0.5 - 0.25j, Cx), (0.5 - 0.25j) * (Cg.conj().T @ Cg)), what + ("complex gram",)
        for k in (40, 72):                            # the TMA-staged update and the parameter-block one
            Y = mx.MxMultiVector(m, 24)
            Y.from_host(Xg[r0:r1])
            Y.MvTimesMatAddMv(0.75, A.CloneView(list(range(k))), B[:k], 2.0)
            assert np.array_equal(Y.to_host(), 0.75 * (Ag[r0:r1, :k] @ B[:k]) + 2.0 * Xg[r0:r1]), what + ("update", k)
        A24 = A.CloneView(list(range(24)))
        assert np.array_equal(X.dot(A24), (Ag[:, :24] * Xg).sum(axis=0)), what + ("dot",)
        assert np.array_equal(Cx.dot(Cx), (np.abs(Cg.real) ** 2 + np.abs(Cg.imag) ** 2).sum(axis=0).astype(complex)), what
        assert np.array_equal(X.norm2(), np.sqrt((Xg * Xg).sum(axis=0))), what + ("norm2",)
        X.remove_const_field()
        assert np.array_equal(X.to_host(), Xg[r0:r1] - Xg.sum(axis=0) * (1.0 / n)), what + ("remove_const_field",)
        del A, X, Cx, A24, Y
    if rank == 0:
        print("case dense block products on ragged partitions ok on %d ranks" % world, flush=True)


def device_assembly_case(ctx, rank, world):
    """Operators assembled on every rank's device (include/mxasm.h), each rank keeping the rows of its slab; the layout is
    built on the device too (ghost discovery, halo plan, dictionary, sliced ELL). Applies must equal the oracle's global
    apply bit for bit, and the layout statistics must be those the same rows give when they come in as host CSR."""
    from maxwell_b200 import assembly as asm
    n = 24
    fine, coarse = asm.example_sim(ctx, "pillbox", n), asm.example_sim(ctx, "pillbox", n // 2)
    of, oc = orc.pillbox(n), orc.pillbox(n // 2)
    maps = {}
    for tag, dsim, osim, nn in (("f", fine, of, n), ("c", coarse, oc, n // 2)):
        for field in ("bfield", "psifield"):
            gids = osim.map(field)
            assert np.array_equal(gids, dsim.map(field))
            cuts = slab_cuts(gids, osim.num_global(field), nn + 1, world)
            maps[tag, field] = (gids, cuts, asm.make_map(dsim, field, cuts[rank], cuts[rank + 1]))

    def check(dop, oop, rkey, ckey, layouts=(0, 1)):
        rg, rcuts, rmap = maps[rkey]
        cg, ccuts, cmap = maps[ckey]
        r0, r1 = rcuts[rank], rcuts[rank + 1]
        rowptr, col, val = oop.arrays()
        lrp, lcol, lval = local_block(rowptr, cg[col], val, r0, r1)
        xg = np.empty((len(cg), 2))
        for j in range(2):
            xg[:, j] = mx.hash_uniform(77, cg, j, 0)
        yg = oop.apply(xg)
        for layout in layouts:
            A = asm.to_crs(dop, rmap, cmap, layout=layout)
            H = mx.MxCrsMatrix.from_csr(rmap, cmap, lrp, lcol, lval, layout=layout)
            assert A.stats() == H.stats(), (A.stats(), H.stats())
            x = mx.MxMultiVector(cmap, 2)
            x.random(77)
            y = mx.MxMultiVector(rmap, 2)
            for rep in range(2):
                A.apply(x, y)
            assert np.array_equal(y.to_host(), yg[r0:r1]), "device-assembled operator differs from the global apply"
            del A, H

    check(fine.op("curlCurl"), of.op("curlCurl"), ("f", "bfield"), ("f", "bfield"))
    check(fine.op("vecLapl"), of.op("vecLapl"), ("f", "bfield"), ("f", "bfield"), layouts=(0,))
    check(fine.op("divB"), of.op("divB"), ("f", "psifield"), ("f", "bfield"), layouts=(0,))
    p = fine.interpolator_from(coarse, "bfield")
    po = orc.interpolator(oc, of)
    check(p, po, ("f", "bfield"), ("c", "bfield"), layouts=(0,))
    check(p.transpose(scale=0.125), po.transpose(scale=0.125), ("c", "bfield"), ("f", "bfield"), layouts=(0,))
    if rank == 0:
        print("case device assembly + device layout ok on %d ranks" % world, flush=True)


def main():
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local_rank = int(os.environ.get("LOCAL_RANK", rank))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    ctx = mx.Context(local_rank)
    ids = [mx.Context.unique_id() if rank == 0 else None]
    dist.broadcast_object_list(ids, src=0)
    ctx.comm_init(rank, world, ids[0])
    assert ctx.myPID() == rank and ctx.numProc() == world

    cases = [("vacuum", orc.vacuum(16), "curlCurl", 1), ("pillbox", orc.pillbox(24), "curlCurl", 3),
             ("pillbox-vecLapl", orc.pillbox(20), "vecLapl", 2),
             ("bloch", orc.vacuum(12, phase_shifts=(0.4, -1.3, 2.2)), "curlCurl", 2)]
    for label, sim, name, nvec in cases:
        n = sim.n[0]
        op = sim.op(name)
        rowptr, col, val = op.arrays()
        rg, _ = op.maps()
        n_global = sim.num_global("bfield")
        cuts = slab_cuts(rg, n_global, n + 1, world)
        r0, r1 = cuts[rank], cuts[rank + 1]
        lrp, lcol, lval = local_block(rowptr, rg[col], val, r0, r1)
        bmap = mx.MxMap(ctx, n_global, rg[r0:r1])
        for layout in (0, 1):
            A = mx.MxCrsMatrix.from_csr(bmap, bmap, lrp, lcol, lval, layout=layout)
            st = A.stats()
            assert st["ghosts"] > 0 and st["ghost_rows"] > 0, (label, st)
            x = mx.MxMultiVector(bmap, nvec, op.is_complex)
            y = mx.MxMultiVector(bmap, nvec, op.is_complex)
            x.random(4242)
            xg = np.empty((len(rg), nvec), dtype=x.dtype)
            for j in range(nvec):
                xg[:, j] = mx.hash_uniform(4242, rg, j, 0)
                if op.is_complex:
                    xg[:, j] += 1j * mx.hash_uniform(4242, rg, j, 1)
            assert np.array_equal(x.to_host(), xg[r0:r1]), "random is not P-invariant"
            for rep in range(3):                      # repeated applies reuse the ghost buffers
                A.apply(x, y)
            yg = op.apply(xg)
            _assert_matches_global(y.to_host(), yg[r0:r1], op.is_complex, (label, layout))
            # the timed apply takes the same path as apply, so it must compute the same y
            ms = A.apply_timed(x, y)
            _assert_matches_global(y.to_host(), yg[r0:r1], op.is_complex, (label, layout, "apply_timed"))
            assert all(0 <= ms[k] <= ms["total_ms"] for k in ("dict_ms", "sell_ms", "pre_ms")), (label, layout, ms)
            if not op.is_complex and os.environ.get("MXG_HALO") != "nccl":
                # default path on one node: the single launch, whose pack and boundary-row roles both run on every rank here
                tl = A.trace_apply(x, y)
                assert -1 not in tl["pack"] and -1 not in tl["boundary_rows"], (label, layout, tl)
            np.testing.assert_allclose(x.norm2(), np.linalg.norm(xg, axis=0), rtol=1e-13)
            np.testing.assert_allclose(y.dot(x), np.einsum("ij,ij->j", xg.conj(), yg), rtol=1e-11, atol=1e-8)
            G = y.MvTransMv(1.0, x)
            np.testing.assert_allclose(G, xg.conj().T @ yg, rtol=1e-10, atol=1e-7)
            del A
        if rank == 0:
            print("case %s ok on %d ranks" % (label, world), flush=True)
    dense_case(ctx, rank, world)
    device_assembly_case(ctx, rank, world)
    solve_case(ctx, rank, world)
    dist.barrier()
    print("RANK %d OK" % rank, flush=True)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()

"""Stand-alone body of tests/test_gpu_spmv.py::test_component_major_ordered_maps (own process: this path had not run on a
GPU when it was written). Operators and vectors on component-major ordered maps (mxg_map_create_ordered) must give exactly
the results of the reference order: bit-exact SpMM for square and rectangular operators (also for an operator assembled on
the device), GID-keyed random vectors, field output, norms / Gram matrices up to summation order, and the same eigenvalues."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    import maxwell_b200 as mx
    from oracle import oracle as orc
    ctx = mx.Context(0)
    sim = orc.pillbox(20)
    fields = {"bfield": 3, "efield": 3, "psifield": 1}
    maps = {f: mx.MxMap(ctx, sim.num_global(f), sim.map(f), components=c) for f, c in fields.items()}
    plain = {f: mx.MxMap(ctx, sim.num_global(f), sim.map(f)) for f in fields}
    assert maps["bfield"].perm is not None and maps["psifield"].perm is None
    ops = {"curlCurl": ("bfield", "bfield"), "vecLapl": ("bfield", "bfield"), "curlE": ("bfield", "efield"),
           "curlB": ("efield", "bfield"), "divB": ("psifield", "bfield"), "gradPsi": ("bfield", "psifield")}
    for name, (rf, cf) in ops.items():
        op = sim.op(name)
        rowptr, col, val = op.arrays()
        rg, cg = op.maps()
        A = mx.MxCrsMatrix.from_csr(maps[rf], maps[cf], rowptr, cg[col], val)
        for nvec in (1, 3):
            x = mx.MxMultiVector(maps[cf], nvec)
            y = mx.MxMultiVector(maps[rf], nvec)
            x.random(4242)
            A.apply(x, y)
            xh = x.to_host()
            assert np.array_equal(op.apply(xh), y.to_host()), (name, nvec)
    # a device-assembled operator on the ordered maps: mxg_crs_create_from_dcsr downloads its rows and lays them out as
    # host CSR, so it must be the operator the oracle's rows make
    from maxwell_b200 import assembly as asm
    op = sim.op("curlCurl")
    rowptr, col, val = op.arrays()
    rg, cg = op.maps()
    A = asm.to_crs(asm.example_sim(ctx, "pillbox", 20).op("curlCurl"), maps["bfield"], maps["bfield"])
    H = mx.MxCrsMatrix.from_csr(maps["bfield"], maps["bfield"], rowptr, cg[col], val)
    assert A.stats() == H.stats(), (A.stats(), H.stats())
    x = mx.MxMultiVector(maps["bfield"], 3)
    x.random(4242)
    ys = []
    for M in (A, H):
        y = mx.MxMultiVector(maps["bfield"], 3)
        M.apply(x, y)
        ys.append(y.to_host())
    assert np.array_equal(ys[0], ys[1]), "device-assembled operator on ordered maps"
    # random vectors are keyed by GID: identical to the reference-order map, column by column
    xo = mx.MxMultiVector(maps["bfield"], 2)
    xp = mx.MxMultiVector(plain["bfield"], 2)
    xo.random(7)
    xp.random(7)
    assert np.array_equal(xo.to_host(), xp.to_host())
    assert np.array_equal(xo.to_host()[:, 1], mx.hash_uniform(7, maps["bfield"].gids, 1, 0))
    # upload / download round trip and field output
    h = np.random.default_rng(0).uniform(-1, 1, (len(maps["bfield"].gids), 2))
    xo.from_host(h)
    assert np.array_equal(xo.to_host(), h)
    total = 3 * 21 ** 3
    want = np.zeros(total)
    want[maps["bfield"].gids] = h[:, 1]
    assert np.array_equal(xo.to_grid(1, 0, total), want)
    # reductions agree up to summation order
    xp.from_host(h)
    np.testing.assert_allclose(xo.norm2(), xp.norm2(), rtol=1e-13)
    np.testing.assert_allclose(xo.trans_mv(1.0, xo), xp.trans_mv(1.0, xp), rtol=1e-12, atol=1e-12)
    # eigenvalues on ordered maps equal the analytic spectrum (periodic vacuum vector Laplacian: each scalar eigenvalue
    # three times), as they do in the reference order
    nv = 10
    vac = orc.vacuum(nv)
    lam1 = (2 * nv * np.sin(np.pi * np.arange(nv) / nv)) ** 2
    scalar = np.sort((lam1[:, None, None] + lam1[None, :, None] + lam1[None, None, :]).ravel())
    want = np.repeat(scalar[:3], 3)[:7]                     # 0 (x3), then the first non-zero eigenvalue
    op = vac.op("vecLapl")
    rowptr, col, val = op.arrays()
    rg, cg = op.maps()
    for comps in (3, 1):
        m = mx.MxMap(ctx, vac.num_global("bfield"), vac.map("bfield"), components=comps)
        A = mx.MxCrsMatrix.from_csr(m, m, rowptr, cg[col], val)
        s = mx.MxSolver(ctx, A, nev=7, block_size=12, tol=1e-9, max_iters=1000)
        ev = s.solve()
        assert s.converged == 7, (comps, s.converged)
        np.testing.assert_allclose(ev[3:7], want[3:7], rtol=1e-8)
        assert np.abs(ev[:3]).max() < 1e-6 * want[3]
    print("ORDERED MAPS OK")


if __name__ == "__main__":
    main()

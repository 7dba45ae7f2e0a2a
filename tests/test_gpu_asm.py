"""Operator assembly on the GPU (SURVEY 8 f2 / f3) against the oracle: cut-cell fractions, DOF maps and every named
operator must come back bit for bit, and an operator assembled on the device must apply exactly like the one uploaded
from the oracle's host CSR. The cases are those of the CPU replay (tests/test_asm_replay.py), which pins the same
sources without a GPU; here the CUDA kernels run.
"""
import numpy as np
import pytest

from test_asm_replay import (CASES, DIELECTRIC_CASES, OPS, both, check_against_independent_fixtures, dielectric_pair,  # noqa: F401
                             pillbox_shape, crabcav_shape, crab_grid)

pytestmark = pytest.mark.gpu


def gpu_pair(asm, ctx, orc, n, origin, size, shape=None, lower=None, upper=None, phase_shifts=None, literal=False,
             use_host_fracs=False):
    api = asm.gpu_api()
    so = sp = None
    if shape is not None:
        so, sp = both(api, shape)
    o = orc.Sim(n, origin=origin, size=size, lower=lower, upper=upper, phase_shifts=phase_shifts, pec=so,
                literal_upper_periodic_e=literal)
    p = asm.gpu_sim(ctx, n, origin=origin, size=size, lower=lower, upper=upper, phase_shifts=phase_shifts,
                    literal_upper_periodic_e=literal)
    if shape is not None:
        if use_host_fracs:
            for f in asm.FIELDS:
                p.set_pec_fractions(f, o.full_fracs(f))
        else:
            p.set_pec_shape(sp)
    p.setup()
    return o, p


@pytest.fixture(scope="module")
def asm(mx):
    from maxwell_b200 import assembly
    return assembly


@pytest.mark.parametrize("case", sorted(CASES))
def test_device_assembly_matches_the_oracle_bit_for_bit(asm, ctx, orc, case):
    o, p = gpu_pair(asm, ctx, orc, **CASES[case])
    for f in asm.FIELDS:
        assert np.array_equal(o.map(f), p.map(f)), f
        ref = o.full_fracs(f)
        if ref is not None:
            got = p.fracs(f)
            bad = np.flatnonzero(ref != got)
            assert bad.size == 0, "%s: %d of %d fractions differ, first %r vs %r" % (f, bad.size, ref.size, ref[bad[:1]], got[bad[:1]])
    for name in OPS:
        a, b = o.op(name), p.op(name)
        assert (a.nrows, a.ncols, a.nnz, a.is_complex) == (b.nrows, b.ncols, b.nnz, b.is_complex), name
        for x, y in zip(a.arrays(), b.arrays()):
            assert np.array_equal(x, y), name


def test_prefix_scan_and_products_at_a_size_that_spans_many_blocks(asm, ctx, orc):
    """40^3 pillbox: 200 k rows, several scan chunks per pass, product rows of every length."""
    o, p = gpu_pair(asm, ctx, orc, 40, (-0.5,) * 3, (1.0,) * 3, shape=pillbox_shape)
    for f in asm.FIELDS:
        assert np.array_equal(o.map(f), p.map(f)), f
        assert np.array_equal(o.full_fracs(f), p.fracs(f)), f
    for name in ("curlCurl", "vecLapl", "scaLapl"):
        for x, y in zip(o.op(name).arrays(), p.op(name).arrays()):
            assert np.array_equal(x, y), name


def test_device_assembled_operator_applies_like_the_uploaded_one(asm, mx, ctx, orc):
    o, p = gpu_pair(asm, ctx, orc, 24, (-0.5,) * 3, (1.0,) * 3, shape=pillbox_shape)
    bmap = asm.make_map(p, "bfield")
    assert np.array_equal(bmap.gids, o.map("bfield"))
    A = asm.to_crs(p.op("curlCurl"), bmap, bmap)
    ref = o.op("curlCurl")
    x = mx.MxMultiVector(bmap, 3)
    x.random(4242)
    y = mx.MxMultiVector(bmap, 3)
    A.apply(x, y)
    assert np.array_equal(ref.apply(x.to_host()), y.to_host())
    st = A.stats()
    assert st["rows"] == ref.nrows and st["nnz"] == ref.nnz and st["dict_rows"] > 0
    # rectangular operator on two maps, sliced-ELL path
    pmap = asm.make_map(p, "psifield")
    D = asm.to_crs(p.op("divB"), pmap, bmap)
    z = mx.MxMultiVector(pmap, 3)
    D.apply(x, z)
    assert np.array_equal(o.op("divB").apply(x.to_host()), z.to_host())


def test_complex_bloch_operator_assembled_on_the_device(asm, mx, ctx, orc):
    o, p = gpu_pair(asm, ctx, orc, **CASES["bloch-pec"])
    bmap = asm.make_map(p, "bfield")
    A = asm.to_crs(p.op("vecLapl"), bmap, bmap)
    x = mx.MxMultiVector(bmap, 2, is_complex=True)
    x.random(99)
    y = mx.MxMultiVector(bmap, 2, is_complex=True)
    A.apply(x, y)
    # complex parity is against the reference's storage, the real 2N K form (MxCrsMatrix.cpp:145-170), as in test_gpu_spmv
    K = o.op("vecLapl").kform()
    xh, got = x.to_host(), y.to_host()
    for j in range(2):
        yk = K.apply(np.ascontiguousarray(xh[:, j]).view(np.float64)).view(np.complex128)
        assert np.array_equal(yk, got[:, j])


def test_dielectric_chain_around_an_uploaded_inverse_permittivity(asm, ctx, orc):
    n = 10
    o = orc.Sim(n, origin=(-0.5,) * 3, size=(1.0,) * 3, pec=orc.Shape.sphere(0.49, (0, 0, 0)),
                dielectrics=[(orc.Shape.sphere(0.37, (0, 0, 0)), orc.SAPPHIRE)])
    api = asm.gpu_api()
    p = asm.gpu_sim(ctx, n, origin=(-0.5,) * 3, size=(1.0,) * 3)
    p.set_pec_shape(api.sphere(0.49, (0, 0, 0))).setup()
    ie, iv = o.op("invEps"), o.op("invEpsVolAve")
    d_ie = p.upload("efield", "efield", *ie.arrays(), ncols=ie.ncols)
    d_iv = p.upload("psifield", "psifield", *iv.arrays(), ncols=iv.ncols)
    for name in ("curlCurl", "vecLapl"):
        for x, y in zip(o.op(name).arrays(), p.op(name, inv_eps=d_ie, inv_eps_vol_ave=d_iv).arrays()):
            assert np.array_equal(x, y), name


def test_errors_are_reported_not_swallowed(asm, ctx):
    api = asm.gpu_api()
    p = asm.gpu_sim(ctx, 6)
    with pytest.raises(asm.AssemblyError):
        p.map("bfield")                      # before setup
    p.setup()
    with pytest.raises(asm.AssemblyError):
        p.op("divB") @ p.op("divB")          # (psi x B) (psi x B): shapes do not chain
    with pytest.raises(asm.AssemblyError):
        api.sim(ctx.h, (0, 4, 4))
    with pytest.raises(asm.AssemblyError):
        api.sim(None, 4)                     # no context: the product never runs without a device


@pytest.mark.parametrize("case", ["pillbox", "vacuum-bloch", "walls"])
def test_grid_transfers_assembled_on_the_device(asm, ctx, orc, case):
    kw = dict(CASES[case])
    n = kw.pop("n")
    n = (n,) * 3 if np.isscalar(n) else n
    fine_n = tuple(2 * (v // 2) for v in n)
    coarse_n = tuple(v // 2 for v in fine_n)
    of, pf = gpu_pair(asm, ctx, orc, n=fine_n, **kw)
    oc, pc = gpu_pair(asm, ctx, orc, n=coarse_n, **kw)
    cx = bool(kw.get("phase_shifts"))
    for field in ("bfield", "psifield"):
        ref = orc.interpolator(oc, of, field=field, is_complex=cx)
        got = pf.interpolator_from(pc, field, is_complex=cx)
        for x, y in zip(ref.arrays(), got.arrays()):
            assert np.array_equal(x, y), field
        for x, y in zip(ref.transpose(scale=0.125).arrays(), got.transpose(scale=0.125).arrays()):
            assert np.array_equal(x, y), field


def test_eigensolve_on_a_problem_assembled_entirely_on_the_device(asm, mx, ctx, orc):
    """Shape -> fractions -> maps -> operators -> hierarchy -> projected eigensolve without a host-generated matrix:
    the 10 lowest Maxwell modes of the 32^3 pillbox against scipy on the ORACLE's curl-curl pencil."""
    from test_gpu_projected import _maxwell_reference
    sizes = [32, 16, 8]
    sims = [asm.example_sim(ctx, "pillbox", n) for n in sizes]
    ep = asm.EigenProblem(ctx, sims)
    prec = mx.MxGeoMultigridPrec(ctx, ep.vops, ep.Rb, ep.Pb, smoother_sweeps=2)
    sprec = mx.MxGeoMultigridPrec(ctx, ep.sops, ep.Rp, ep.Pp, smoother_sweeps=2, remove_const_field=True)
    nev = 10
    s = mx.MxSolver(ctx, ep.vops[0], m_diag=ep.m_diag, prec=prec, nev=nev, block_size=16, tol=1e-9, max_iters=300,
                    projection={"divB": ep.divB, "gradPsi": ep.gradPsi, "scaLapl": ep.sops[0], "sca_prec": sprec})
    ev = s.solve()
    assert s.converged == nev, (s.converged, s.residuals)
    ref = _maxwell_reference(orc.pillbox(32), nev, sigma=60.0)
    np.testing.assert_allclose(ev, ref, rtol=1e-9)
    res, div = s.check(ep.divB, A=ep.curlCurl)
    assert np.all(res[:nev] < 1e-6) and np.all(div[:nev] < 1e-6)


@pytest.mark.parametrize("case,name", [("pillbox", "curlCurl"), ("pillbox", "vecLapl"), ("pillbox", "divB"), ("crabcav", "curlCurl"),
                                       ("bloch-pec", "vecLapl"), ("vacuum", "curlCurl")])
def test_host_and_device_rows_make_the_same_layout(asm, mx, ctx, orc, case, name):
    """The oracle's host CSR (mxg_crs_create) and the device-assembled rows (mxg_crs_create_from_dcsr) reach the same
    layout: the same statistics, which follow the single-rank layout rules restated in numpy, and bit-identical applies."""
    from conftest import gpu_matrix
    kw = dict(CASES[case])
    if case == "pillbox":
        kw["n"] = 20
    o, p = gpu_pair(asm, ctx, orc, **kw)
    H, op, rmap, cmap = gpu_matrix(mx, ctx, o, name)
    rf, cf = {"curlCurl": ("bfield", "bfield"), "vecLapl": ("bfield", "bfield"), "divB": ("psifield", "bfield")}[name]
    dr = asm.make_map(p, rf)
    dc = dr if rf == cf else asm.make_map(p, cf)
    d = p.op(name)
    for layout in (0, 1):
        Hl = mx.MxCrsMatrix.from_csr(rmap, cmap, *_global(op), layout=layout)
        A = asm.to_crs(d, dr, dc, layout=layout)
        assert A.stats() == Hl.stats(), (layout, A.stats(), Hl.stats())
        got = {k: v for k, v in A.stats().items() if k != "device_bytes"}
        want = _layout_reference(op, square=rf == cf, layout=layout)
        assert got == want, (layout, got, want)
        x = mx.MxMultiVector(dc, 3, is_complex=op.is_complex)
        x.random(31)
        ys = []
        for M in (A, Hl):
            y = mx.MxMultiVector(dr, 3, is_complex=op.is_complex)
            M.apply(x, y)
            ys.append(y.to_host())
        assert np.array_equal(ys[0], ys[1]), layout
    assert H.stats()["rows"] == d.nrows


def test_domain_map_that_is_not_a_run_of_the_field_map(asm, mx, ctx, orc):
    """A domain map that is not a contiguous run of the column field's map (here every GID of the B field's space) sends
    mxg_crs_create_from_dcsr through its download route: the rows come to the host and mxg_crs_create lays them out, so
    the operator must be the one the oracle's rows make on the same two maps."""
    o, p = orc.pillbox(20), asm.example_sim(ctx, "pillbox", 20)
    op = o.op("curlCurl")
    bmap = asm.make_map(p, "bfield")
    n = o.num_global("bfield")
    assert len(bmap.gids) < n
    dense = mx.MxMap(ctx, n, np.arange(n))
    for layout in (0, 1):
        A = asm.to_crs(p.op("curlCurl"), bmap, dense, layout=layout)
        H = mx.MxCrsMatrix.from_csr(bmap, dense, *_global(op), layout=layout)
        assert A.stats() == H.stats(), (layout, A.stats(), H.stats())
        x = mx.MxMultiVector(dense, 3)
        x.random(4242)
        ys = []
        for M in (A, H):
            y = mx.MxMultiVector(bmap, 3)
            M.apply(x, y)
            ys.append(y.to_host())
        assert np.array_equal(ys[0], ys[1]), layout
        assert np.array_equal(ys[0], op.apply(x.to_host()[op.maps()[1]])), layout


def _global(op):
    rowptr, col, val = op.arrays()
    _, cg = op.maps()
    return rowptr, cg[col], val


def _layout_reference(op, square, layout):
    """Statistics of the single-rank layout of an oracle operator: with layout 0 on a square operator, a non-empty row's
    key is (length, column - row of every entry, value bytes) and every key seen at least 4 times is a dictionary
    pattern; the remaining rows go to sliced ELL in groups of 32 consecutive rows, each as wide as its longest row."""
    rowptr, col, val = op.arrays()
    n = len(rowptr) - 1
    lens = np.diff(rowptr)
    counts, key_of = {}, [None] * n
    if layout == 0 and square:
        for r in range(n):
            b, e = rowptr[r], rowptr[r + 1]
            if b == e:
                continue
            assert np.all(np.diff(col[b:e]) > 0), "rows must be sorted and merged"
            key_of[r] = (int(e - b), (col[b:e].astype(np.int64) - r).tobytes(), val[b:e].tobytes())
            counts[key_of[r]] = counts.get(key_of[r], 0) + 1
    frequent = {k: c for k, c in counts.items() if c >= 4}
    rest = np.array([lens[r] for r in range(n) if key_of[r] not in frequent], dtype=np.int64)
    rest = np.concatenate([rest, np.zeros(-len(rest) % 32, dtype=np.int64)])
    return {"rows": n, "nnz": int(rowptr[-1]), "dict_rows": sum(frequent.values()), "patterns": len(frequent),
            "ghosts": 0, "ghost_rows": 0, "ell_entries": 32 * int(rest.reshape(-1, 32).max(axis=1).sum())}


def test_smoothers_see_the_same_inverse_diagonal(asm, mx, ctx, orc):
    """The V-cycle uses 1 / diag(A) kept with the operator: one multigrid application must give identical bits whether
    the level operators and transfers come in as device rows or as host CSR (the same rows, downloaded)."""
    sizes = [16, 8]
    sims = [asm.example_sim(ctx, "pillbox", n) for n in sizes]
    ep = asm.EigenProblem(ctx, sims)
    gids = [s.map("bfield") for s in sims]

    def from_host(d, rl, cl):
        rowptr, col, val = d.arrays()
        return mx.MxCrsMatrix.from_csr(ep.bmaps[rl], ep.bmaps[cl], rowptr, gids[cl][col], val)

    p = sims[0].interpolator_from(sims[1], "bfield")
    host = ([from_host(s.op("vecLapl"), l, l) for l, s in enumerate(sims)], [from_host(p.transpose(scale=0.125), 1, 0)],
            [from_host(p, 0, 1)])
    outs = []
    for vops, Rb, Pb in ((ep.vops, ep.Rb, ep.Pb), host):
        prec = mx.MxGeoMultigridPrec(ctx, vops, Rb, Pb, smoother_sweeps=2)
        b = mx.MxMultiVector(ep.bmaps[0], 2)
        b.random(8)
        x = b.Clone(2)
        prec.ApplyInverse(b, x)
        outs.append(x.to_host())
    assert np.array_equal(outs[0], outs[1])


@pytest.mark.parametrize("case", sorted(DIELECTRIC_CASES))
def test_inverse_permittivity_assembled_on_the_device(asm, mx, ctx, orc, case):
    """MxYeeFitInvEps on the device: anisotropic 9-point rows (3x3 complex inversions with libgcc's division order,
    interface normals from the shape gradient), the scalar cell average, and the chains through them -- bit for bit."""
    kw = DIELECTRIC_CASES[case]
    o, p = dielectric_pair(lambda n, **k: asm.gpu_sim(ctx, n, **k), asm.gpu_api(), **kw)
    cx = bool(kw.get("phase_shifts")) or any(np.iscomplexobj(e) for _, e in kw["diels"])
    for name in ("invEps", "invEpsVolAve", "curlCurl", "gradDiv", "vecLapl"):
        a, b = o.op(name, is_complex=cx), p.op(name, is_complex=cx)
        assert (a.nrows, a.ncols, a.nnz) == (b.nrows, b.ncols, b.nnz), name
        for x, y in zip(a.arrays(), b.arrays()):
            bad = np.flatnonzero(x != y)
            assert bad.size == 0, "%s: %d of %d entries differ, first %r vs %r" % (name, bad.size, x.size, x[bad[:1]], y[bad[:1]])
    # and the assembled operator applies like the oracle's (K-form order when complex)
    bmap = asm.make_map(p, "bfield")
    A = asm.to_crs(p.op("vecLapl", is_complex=cx), bmap, bmap)
    x = mx.MxMultiVector(bmap, 2, is_complex=cx)
    x.random(5)
    y = mx.MxMultiVector(bmap, 2, is_complex=cx)
    A.apply(x, y)
    ref = o.op("vecLapl", is_complex=cx)
    xh, got = x.to_host(), y.to_host()
    if cx:
        K = ref.kform()
        for j in range(2):
            assert np.array_equal(K.apply(np.ascontiguousarray(xh[:, j]).view(np.float64)).view(np.complex128), got[:, j])
    else:
        assert np.array_equal(ref.apply(xh), got)


def test_device_assembly_against_fixtures_independent_of_the_oracle(asm, ctx):
    """The scipy Kronecker-product vacuum curl-curl and the analytic vacuum spectrum of tests/golden/ (no code shared with
    the oracle), plus div curl = 0 and curlCurl grad = 0 on the cut-cell pillbox."""
    check_against_independent_fixtures(lambda n, **k: asm.gpu_sim(ctx, n, **k))

"""Slab-partitioned operator assembly (include/mxasm.h: mxg_sim_op_rows, mxg_sim_interpolator_rows,
mxg_sim_interpolator_transpose_rows) on the CPU replay of the assembly sources.

A rank that owns the rows [r0, r1) of an operator's row map assembles only those rows: each chain factor on the rows its
left neighbour references, the products in the reference's association order. The rows must equal the rows [r0, r1)
of the whole-map operator bit for bit, for every named operator, grid transfer and restriction, on the x-slabs of 2, 3
and 8 ranks, on periodic-x grids (where rank 0 reaches the top planes) and for ranges that are not slabs at all.
tests/test_gpu_asm_slab.py runs the same checks on the device.
"""
import numpy as np
import pytest

from maxwell_b200 import assembly as asm
from maxwell_b200.partition import slab_cuts
from test_asm_replay import CASES, DIELECTRIC_CASES, OPS, api, dielectric_pair, make_pair  # noqa: F401

SLAB_CASES = ("pillbox", "crabcav", "tilted", "walls", "walls-mixed", "vacuum", "vacuum-bloch", "bloch-pec")
WORLDS = (2, 3, 8)
ROW_FIELD = {"curlE": "bfield", "curlB": "efield", "divB": "psifield", "gradPsi": "bfield", "dmA": "bfield", "dmL": "efield",
             "dmVInv": "psifield", "mRhs": "bfield", "invEps": "efield", "invEpsVolAve": "psifield", "curlCurl": "bfield",
             "gradDiv": "bfield", "vecLapl": "bfield", "scaLapl": "psifield"}


def row_ranges(sim, field, worlds=WORLDS):
    """The x-slabs of every rank of every world, then an empty range, a single row, a range that does not start on a plane
    boundary, and the whole map."""
    gids = sim.map(field)
    n = len(gids)
    out = []
    for w in worlds:
        cuts = slab_cuts(gids, sim.num_global(field), sim.n[0] + 1, w)
        out += list(zip(cuts[:-1], cuts[1:]))
    out += [(n // 2, n // 2), (max(n - 1, 0) // 3, max(n - 1, 0) // 3 + 1), (n // 3 + 1, (2 * n) // 3 + 2), (0, n)]
    return [(int(a), int(min(b, n))) for a, b in out if a <= min(b, n)]


def assert_rows_equal(whole, part, r0, r1, what):
    assert (part.row_begin, part.nrows, part.ncols, part.is_complex) == (r0, r1 - r0, whole.ncols, whole.is_complex), what
    assert (part.row_field, part.col_field) == (whole.row_field, whole.col_field), what
    rp, col, val = whole.arrays()
    prp, pcol, pval = part.arrays()
    assert np.array_equal(prp, rp[r0:r1 + 1] - rp[r0]), what + ("rowptr",)
    assert np.array_equal(pcol, col[rp[r0]:rp[r1]]), what + ("col",)
    assert np.array_equal(pval, val[rp[r0]:rp[r1]]), what + ("val",)


def check_operator_rows(sim, names, is_complex=None, worlds=WORLDS):
    for name in names:
        whole = sim.op(name, is_complex)
        for r0, r1 in row_ranges(sim, ROW_FIELD[name], worlds):
            assert_rows_equal(whole, sim.op(name, is_complex, rows=(r0, r1)), r0, r1, (name, r0, r1))


def check_transfer_rows(fine, coarse, is_complex, worlds=WORLDS):
    """Interpolator rows on the fine map and restriction rows on the coarse map against the whole P and P^H."""
    for field in ("bfield", "psifield"):
        p = fine.interpolator_from(coarse, field, is_complex)
        for r0, r1 in row_ranges(fine, field, worlds):
            assert_rows_equal(p, fine.interpolator_from(coarse, field, is_complex, rows=(r0, r1)), r0, r1, ("P", field, r0, r1))
        t = p.transpose()
        for r0, r1 in row_ranges(coarse, field, worlds):
            assert_rows_equal(t, fine.interpolator_transpose(coarse, field, is_complex, rows=(r0, r1)), r0, r1, ("R", field, r0, r1))
        assert_rows_equal(t.scale(0.125), fine.interpolator_transpose(coarse, field, is_complex).scale(0.125), 0, t.nrows, ("R/8", field))


def transfer_pair(new_sim, case):
    kw = dict(CASES[case])
    n = kw.pop("n")
    n = (n,) * 3 if np.isscalar(n) else n
    fine_n = tuple(2 * (v // 2) for v in n)
    return new_sim(fine_n, kw), new_sim(tuple(v // 2 for v in fine_n), kw), bool(kw.get("phase_shifts"))


@pytest.mark.parametrize("case", SLAB_CASES)
def test_operator_rows_equal_the_rows_of_the_whole_operator(api, case):
    _, p = make_pair(api, **CASES[case])
    check_operator_rows(p, OPS)


@pytest.mark.parametrize("case", ["pillbox", "vacuum", "vacuum-bloch", "walls"])
def test_transfer_and_restriction_rows_equal_those_of_the_whole_transfer(api, case):
    fine, coarse, cx = transfer_pair(lambda n, kw: make_pair(api, n=n, **kw)[1], case)
    check_transfer_rows(fine, coarse, cx)


@pytest.mark.parametrize("case", ["dsphmsph", "phc-sapphire"])
def test_dielectric_operator_rows(api, case):
    kw = DIELECTRIC_CASES[case]
    _, p = dielectric_pair(lambda n, **k: api.sim(None, n, **k), api, **kw)
    cx = bool(kw.get("phase_shifts")) or any(np.iscomplexobj(e) for _, e in kw["diels"])
    check_operator_rows(p, ("invEps", "invEpsVolAve", "curlCurl", "gradDiv", "vecLapl", "scaLapl"), is_complex=cx)


def test_handed_in_dielectric_factors_whole_or_partial(api):
    kw = DIELECTRIC_CASES["dsphmsph"]
    _, p = dielectric_pair(lambda n, **k: api.sim(None, n, **k), api, **kw)
    ie, iv = p.op("invEps"), p.op("invEpsVolAve")
    whole = p.op("vecLapl")
    n = whole.nrows
    r0, r1 = row_ranges(p, "bfield", (3,))[1]
    assert_rows_equal(whole, p.op("vecLapl", inv_eps=ie, inv_eps_vol_ave=iv, rows=(r0, r1)), r0, r1, ("given whole",))
    # partial factors that store exactly what a slab needs are accepted: here the E / psi rows of the middle third and more
    ne, npsi = ie.nrows, iv.nrows
    part_e = p.op("invEps", rows=(ne // 6, ne - ne // 6))
    part_v = p.op("invEpsVolAve", rows=(npsi // 6, npsi - npsi // 6))
    assert part_e.row_begin == ne // 6
    mid = (n // 2 - n // 20, n // 2 + n // 20)
    assert_rows_equal(whole, p.op("vecLapl", inv_eps=part_e, inv_eps_vol_ave=part_v, rows=mid), *mid, ("given partial",))
    # ... and a factor that lacks rows the chain needs is an error, not a short or wrong row
    with pytest.raises(asm.AssemblyError, match="no stored row"):
        p.op("curlCurl", inv_eps=p.op("invEps", rows=(0, 1)), rows=mid)


def test_the_crs_algebra_takes_partial_operands_under_the_covering_rules(api):
    _, p = make_pair(api, **CASES["vacuum"])
    nb = p.map_size("bfield")[0]
    r0, r1 = row_ranges(p, "bfield", (3,))[1]
    ce, cb = p.op("curlE", rows=(r0, r1)), p.op("curlB")
    assert_rows_equal(p.op("curlE") @ cb, ce @ cb, r0, r1, ("partial A, whole B",))
    # B partial but storing every row A references: the E rows of the slab's planes +- one plane, wrapping around
    ne = p.map_size("efield")[0]
    cb_part = p.op("curlB", rows=(0, ne))
    assert_rows_equal(p.op("curlE") @ cb, ce @ cb_part, r0, r1, ("partial A, covering B",))
    with pytest.raises(asm.AssemblyError, match="no stored row in B"):
        ce @ p.op("curlB", rows=(0, 1))
    cc = p.op("curlCurl", rows=(r0, r1))
    gd = p.op("gradDiv", rows=(r0, r1))
    assert_rows_equal(p.op("vecLapl"), cc.add(1.0, gd, -1.0, purge=True), r0, r1, ("add",))
    assert_rows_equal(p.op("vecLapl"), cc.add(1.0, p.op("gradDiv"), -1.0, purge=True), r0, r1, ("add, whole B",))
    with pytest.raises(asm.AssemblyError):
        p.op("gradDiv").add(1.0, cc, -1.0)                  # B lacks A's rows
    with pytest.raises(asm.AssemblyError, match="interpolator_transpose_rows"):
        ce.transpose()
    assert p.op("curlE", rows=(0, nb)).transpose().nrows == ne


def test_misuse_returns_an_error_code(api):
    _, p = make_pair(api, **CASES["pillbox"])
    nb, npsi = p.map_size("bfield")[0], p.map_size("psifield")[0]
    for rows in ((5, 3), (0, nb + 1), (-1, 2), (nb + 1, nb + 2)):
        with pytest.raises(asm.AssemblyError, match="range"):
            p.op("curlCurl", rows=rows)
    with pytest.raises(asm.AssemblyError, match="range"):
        p.op("scaLapl", rows=(0, npsi + 1))
    with pytest.raises(asm.AssemblyError, match="unknown operator"):
        p.op("noSuchOperator", rows=(0, 1))
    _, q = make_pair(api, n=6, origin=(-0.5,) * 3, size=(1.0,) * 3, shape=asm.pillbox_shape)
    nq = q.map_size("bfield")[0]
    with pytest.raises(asm.AssemblyError, match="range"):
        api.sim(None, 12, origin=(-0.5,) * 3, size=(1.0,) * 3).setup().interpolator_from(q, "bfield", rows=(3, 2))
    f = make_pair(api, n=12, origin=(-0.5,) * 3, size=(1.0,) * 3, shape=asm.pillbox_shape)[1]
    with pytest.raises(asm.AssemblyError, match="range"):
        f.interpolator_transpose(q, "bfield", rows=(0, nq + 1))
    with pytest.raises(asm.AssemblyError, match="range"):
        f.interpolator_from(q, "bfield", rows=(0, nb + 1))

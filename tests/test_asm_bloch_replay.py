"""Bloch-consistent grid transfers (include/mxasm.h: MXG_INTERP_BLOCH, DESIGN.md GMG-bloch) on the CPU replay of the
assembly sources, against the oracle bit for bit.

With the flag, a stencil cell of the trilinear interpolator that wraps across a periodic face of the coarse grid carries
that direction's Bloch factor: e^{+i phi} from the top, e^{-i phi} from below. The replayed device code must equal the
oracle's restatement to the last bit (values compared as raw bytes, so even the sign of a zero counts) for B and psi
transfers, whole, on row windows and on the restriction windows of x-slabs, including rank 0's window whose fine rows
wrap around a periodic x axis. With all phases 0 the flag must change nothing, and a real transfer of a problem with a
non-zero phase must be refused. tests/test_gpu_bloch.py repeats the comparison on the device.
"""
import numpy as np
import pytest

import bloch_oracle as BO
from oracle import oracle as orc
from maxwell_b200 import assembly as asm
from test_asm_replay import CASES, DIELECTRIC_CASES, api, dielectric_pair, make_pair  # noqa: F401
from test_asm_slab_replay import row_ranges

FIELDS = ("bfield", "psifield")

# periodic y with a Bloch phase between PEC / PMC walls on x and z
WALLS_MIXED_BLOCH = dict(CASES["walls-mixed"], phase_shifts=(0.0, 0.8, 0.0))
BLOCH_CASES = {
    "vacuum-bloch": CASES["vacuum-bloch"],
    "bloch-pec": CASES["bloch-pec"],
    "walls-mixed-bloch": WALLS_MIXED_BLOCH,
}


def halves(n):
    n = (n,) * 3 if np.isscalar(n) else tuple(n)
    fine = tuple(2 * (v // 2) for v in n)
    return fine, tuple(v // 2 for v in fine)


def transfer_pairs(api, case):
    """(oracle fine, oracle coarse, replay fine, replay coarse) of a grid and the one with half the cells."""
    if case == "phc-sapphire":
        kw = dict(DIELECTRIC_CASES[case])
        fine_n, coarse_n = halves(kw.pop("n"))
        of, pf = dielectric_pair(lambda n, **k: api.sim(None, n, **k), api, n=fine_n, **kw)
        oc, pc = dielectric_pair(lambda n, **k: api.sim(None, n, **k), api, n=coarse_n, **kw)
        return of, oc, pf, pc
    kw = dict(BLOCH_CASES[case])
    fine_n, coarse_n = halves(kw.pop("n"))
    of, pf = make_pair(api, n=fine_n, **kw)
    oc, pc = make_pair(api, n=coarse_n, **kw)
    return of, oc, pf, pc


def same_bits(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    return a.dtype == b.dtype and a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def assert_same(ref, got, what):
    assert (ref.nrows, ref.ncols, ref.nnz) == (got.nrows, got.ncols, got.nnz), what
    for x, y in zip(ref.arrays(), got.arrays()):
        assert same_bits(x, y), what


def assert_rows(whole, part, r0, r1, what):
    assert (part.row_begin, part.nrows, part.ncols) == (r0, r1 - r0, whole.ncols), what
    rp, col, val = whole.arrays()
    prp, pcol, pval = part.arrays()
    assert np.array_equal(prp, rp[r0:r1 + 1] - rp[r0]), what
    assert np.array_equal(pcol, col[rp[r0]:rp[r1]]), what
    assert same_bits(pval, val[rp[r0]:rp[r1]]), what


def check_bloch_transfers(api, case):
    """The whole P, P^H and P^H / 8 of both fields, and their row windows, against the oracle (api: the replay or the device)."""
    of, oc, pf, pc = transfer_pairs(api, case)
    for field in FIELDS:
        ref = BO.interpolator(oc, of, field=field, is_complex=True, bloch=True)
        got = pf.interpolator_from(pc, field, True, bloch=True)
        assert_same(ref, got, (case, field, "P"))
        plain = pf.interpolator_from(pc, field, True)
        assert not same_bits(plain.arrays()[2], got.arrays()[2]), "the flag changed nothing on a Bloch-periodic grid"
        rt = ref.transpose()
        gt = pf.interpolator_transpose(pc, field, True, bloch=True)
        assert_same(rt, gt, (case, field, "P^H"))
        assert_same(ref.transpose(scale=0.125), got.transpose(scale=0.125), (case, field, "P^H / 8"))
        # row windows of P (fine map) and of P^H (coarse map): the x-slabs of 2, 3 and 8 ranks and ranges off the planes
        for r0, r1 in row_ranges(pf, field):
            assert_rows(got, pf.interpolator_from(pc, field, True, rows=(r0, r1), bloch=True), r0, r1, (case, field, "P", r0, r1))
        for r0, r1 in row_ranges(pc, field):
            assert_rows(gt, pf.interpolator_transpose(pc, field, True, rows=(r0, r1), bloch=True), r0, r1,
                        (case, field, "P^H", r0, r1))


@pytest.mark.parametrize("case", sorted(BLOCH_CASES) + ["phc-sapphire"])
def test_bloch_transfers_match_the_oracle_bit_for_bit(api, case):
    check_bloch_transfers(api, case)


def test_rank0_restriction_window_wraps_on_periodic_x(api):
    """On a periodic-x grid the fine rows that reach rank 0's coarse planes include the top fine planes, whose stencils wrap
    around to coarse plane 0 with the factor e^{+i phi_x}: the window must hold them, with that factor."""
    of, oc, pf, pc = transfer_pairs(api, "vacuum-bloch")
    from maxwell_b200.partition import slab_cuts
    for field in FIELDS:
        ref = BO.interpolator(oc, of, field=field, is_complex=True, bloch=True).transpose()
        cuts = slab_cuts(pc.map(field), pc.num_global(field), pc.n[0] + 1, 2)
        r0, r1 = int(cuts[0]), int(cuts[1])
        part = pf.interpolator_transpose(pc, field, True, rows=(r0, r1), bloch=True)
        rp, col, val = ref.arrays()
        prp, pcol, pval = part.arrays()
        assert np.array_equal(prp, rp[r0:r1 + 1] - rp[r0]) and np.array_equal(pcol, col[rp[r0]:rp[r1]])
        assert same_bits(pval, val[rp[r0]:rp[r1]])
        top = of.map(field) // (of.num_global(field) // (of.n[0] + 1)) >= of.n[0] - 1
        assert np.any(top[pcol]), "rank 0's restriction rows do not reach the top fine planes"
        assert np.any(np.abs(pval.imag) > 1e-3), "no Bloch factor in rank 0's window"


@pytest.mark.parametrize("case", ["vacuum", "pillbox", "walls-mixed", "bloch-pec-zero"])
def test_flag_with_zero_phases_equals_the_plain_transfer(api, case):
    kw = dict(CASES["bloch-pec"], phase_shifts=(0.0, 0.0, 0.0)) if case == "bloch-pec-zero" else dict(CASES[case])
    fine_n, coarse_n = halves(kw.pop("n"))
    of, pf = make_pair(api, n=fine_n, **kw)
    oc, pc = make_pair(api, n=coarse_n, **kw)
    for field in FIELDS:
        for cx in (False, True):
            plain = pf.interpolator_from(pc, field, cx)
            assert_same(plain, pf.interpolator_from(pc, field, cx, bloch=True), (case, field, cx))
            assert_same(pf.interpolator_transpose(pc, field, cx), pf.interpolator_transpose(pc, field, cx, bloch=True), (case, field, cx))
            assert_same(orc.interpolator(oc, of, field=field, is_complex=cx),
                        BO.interpolator(oc, of, field=field, is_complex=cx, bloch=True), (case, field, cx, "oracle"))


def test_real_bloch_transfer_with_a_phase_is_refused(api):
    _, _, pf, pc = transfer_pairs(api, "vacuum-bloch")
    n = pf.map_size("bfield")[0]
    with pytest.raises(asm.AssemblyError, match="complex"):
        pf.interpolator_from(pc, "bfield", False, bloch=True)
    with pytest.raises(asm.AssemblyError, match="complex"):
        pf.interpolator_from(pc, "bfield", False, rows=(0, n // 2), bloch=True)
    with pytest.raises(asm.AssemblyError, match="complex"):
        pf.interpolator_transpose(pc, "psifield", False, bloch=True)
    # the plain real transfer of the same grids stays available (it is what a real build of a Bloch problem used before)
    assert pf.interpolator_from(pc, "bfield", False).nnz > 0


def test_bloch_transfer_between_different_phases_is_refused(api):
    kw = dict(CASES["vacuum-bloch"])
    fine_n, coarse_n = halves(kw.pop("n"))
    _, pf = make_pair(api, n=fine_n, **kw)
    _, pc = make_pair(api, n=coarse_n, **dict(kw, phase_shifts=(0.3, -0.7, 1.2)))
    with pytest.raises(asm.AssemblyError, match="phase"):
        pf.interpolator_from(pc, "bfield", True, bloch=True)
    lib = api.lib
    import ctypes as C
    h = C.c_void_p()
    assert lib.mxr_sim_interpolator_ex(pc.handle, pf.handle, b"bfield", 1, 2, C.byref(h)) != 0    # unknown flag bit


def test_constant_null_vector_helper(api):
    s = lambda **kw: api.sim(None, 4, **kw)
    assert asm.scalar_laplacian_has_constant_null_vector(s())
    assert asm.scalar_laplacian_has_constant_null_vector(s(phase_shifts=(2.0 * np.pi, 0.0, -4.0 * np.pi)))
    assert not asm.scalar_laplacian_has_constant_null_vector(s(phase_shifts=(0.0, 0.0, 2.0 * np.pi / 3.0)))
    assert not asm.scalar_laplacian_has_constant_null_vector(s(phase_shifts=(2.0, 1.1, 0.4)))
    assert asm.scalar_laplacian_has_constant_null_vector(s(lower=(orc.PEC, 0, 0), upper=(orc.PEC, 0, 0)))
    assert not asm.scalar_laplacian_has_constant_null_vector(s(lower=(orc.PMC, 0, 0), upper=(orc.PEC, 0, 0)))
    # a phase on a non-periodic direction does nothing
    assert asm.scalar_laplacian_has_constant_null_vector(s(lower=(orc.PEC, 0, 0), upper=(orc.PEC, 0, 0), phase_shifts=(0.5, 0, 0)))

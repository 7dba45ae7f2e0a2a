"""Slab-partitioned operator assembly on the GPU (include/mxasm.h: mxg_sim_op_rows, mxg_sim_interpolator_rows,
mxg_sim_interpolator_transpose_rows, mxg_asm_memory): the rows of a rank's x-slab, assembled from the rows its chains
reach only, equal the rows of the whole-map operators bit for bit, lay out and apply like them, and take a fraction of
the assembly memory. tests/test_asm_slab_replay.py pins the same sources on the CPU.
"""
import numpy as np
import pytest

from test_asm_replay import CASES, OPS
from test_asm_slab_replay import assert_rows_equal, check_operator_rows, check_transfer_rows, row_ranges

pytestmark = pytest.mark.gpu
WORLDS = (2, 8)
PHC_PHASES = (2.0, 1.1, 0.4)


@pytest.fixture(scope="module")
def asm(mx):
    from maxwell_b200 import assembly
    return assembly


def walls_sim(asm, ctx, n=None):
    kw = dict(CASES["walls"])
    shape = kw.pop("shape")
    kw.pop("n")
    p = asm.gpu_sim(ctx, n or (12, 10, 14), **kw)
    p.set_pec_shape(shape(asm.gpu_api()))
    return p.setup()


def make(asm, ctx, case, n):
    if case == "walls":
        return walls_sim(asm, ctx, n)
    return asm.example_sim(ctx, case, n, phase_shifts=PHC_PHASES if case == "phc" else None)


@pytest.mark.parametrize("case,n", [("pillbox", 32), ("crabcav", 20), ("dsphmsph", 16), ("phc", 12), ("walls", None)])
def test_slab_rows_equal_the_rows_of_the_whole_operators(asm, ctx, case, n):
    p = make(asm, ctx, case, n)
    names = OPS + (("invEps", "invEpsVolAve") if case in ("dsphmsph", "phc") else ())
    check_operator_rows(p, names, is_complex=True if case == "phc" else None, worlds=WORLDS)


@pytest.mark.parametrize("case,n", [("pillbox", 32), ("phc", 12), ("walls", (12, 10, 14))])
def test_slab_transfer_and_restriction_rows(asm, ctx, case, n):
    nn = (n,) * 3 if np.isscalar(n) else n
    fine, coarse = make(asm, ctx, case, nn), make(asm, ctx, case, tuple(v // 2 for v in nn))
    check_transfer_rows(fine, coarse, case == "phc", worlds=WORLDS)


@pytest.mark.parametrize("case,name", [("pillbox", "vecLapl"), ("pillbox", "divB"), ("phc", "curlCurl")])
def test_whole_range_operator_applies_like_the_whole_operator(asm, mx, ctx, case, name):
    p = make(asm, ctx, case, 24 if case == "pillbox" else 12)
    cx = case == "phc"
    rf, cf = {"vecLapl": ("bfield", "bfield"), "curlCurl": ("bfield", "bfield"), "divB": ("psifield", "bfield")}[name]
    rmap = asm.make_map(p, rf)
    cmap = rmap if rf == cf else asm.make_map(p, cf)
    ys = []
    for d in (p.op(name, cx), p.op(name, cx, rows=(0, p.map_size(rf)[0]))):
        A = asm.to_crs(d, rmap, cmap)
        x = mx.MxMultiVector(cmap, 3, is_complex=cx)
        x.random(17)
        y = mx.MxMultiVector(rmap, 3, is_complex=cx)
        A.apply(x, y)
        ys.append(y.to_host())
    assert np.array_equal(ys[0], ys[1])


def test_assembly_memory_of_a_middle_slab(asm, ctx):
    """vecLapl of one middle rank of world 8 on pillbox-128: the peak assembly bytes above the post-setup baseline are at
    most 0.3 of those of the whole-map build (16 planes + the chains' reach of at most 2 planes per side ~ 0.2 of the map)."""
    p = asm.example_sim(ctx, "pillbox", 128)
    r0, r1 = row_ranges(p, "bfield", (8,))[3]
    peaks = {}
    for label, rows in (("slab", (r0, r1)), ("whole", None)):
        base, _ = asm.asm_memory(ctx, reset_peak=True)
        d = p.op("vecLapl", rows=rows)
        peaks[label] = asm.asm_memory(ctx)[1] - base
        del d
    ratio = peaks["slab"] / peaks["whole"]
    print("pillbox-128 vecLapl assembly peak above baseline: slab %d B, whole %d B, ratio %.3f" % (peaks["slab"], peaks["whole"], ratio))
    assert ratio <= 0.3, peaks
    cur, _ = asm.asm_memory(ctx, reset_peak=True)
    assert cur == base, "the assembly's temporaries and matrices are released"


def test_slab_of_a_rank_on_an_empty_or_single_row_range(asm, ctx):
    p = asm.example_sim(ctx, "pillbox", 16)
    whole = p.op("curlCurl")
    n = whole.nrows
    for r0, r1 in ((0, 0), (n, n), (n - 1, n), (7, 8)):
        assert_rows_equal(whole, p.op("curlCurl", rows=(r0, r1)), r0, r1, (r0, r1))
    with pytest.raises(asm.AssemblyError):
        p.op("curlCurl", rows=(3, 2))
    with pytest.raises(asm.AssemblyError, match="interpolator_transpose_rows"):
        p.op("curlCurl", rows=(0, 5)).transpose()

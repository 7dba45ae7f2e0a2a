"""GPU parity: mxg_crs_apply through the C ABI vs the oracle's Epetra-order CSR apply.
Bar (north_star): 1e-12 relative 2-norm; these kernels are bit-exact, which is what we assert."""
import numpy as np
import pytest

from conftest import gpu_matrix, rel_err

pytestmark = pytest.mark.gpu


def _apply_case(mx, ctx, orc, sim, name, nvec, layout, is_complex=None):
    A, op, rmap, cmap = gpu_matrix(mx, ctx, sim, name, layout=layout, is_complex=is_complex)
    x = mx.MxMultiVector(cmap, nvec, op.is_complex)
    y = mx.MxMultiVector(rmap, nvec, op.is_complex)
    x.random(777)
    y.set(123.0)                      # apply must overwrite, not accumulate
    A.apply(x, y)
    ref = op.apply(x.to_host())
    got = y.to_host()
    return A, op, ref, got, x, y


@pytest.mark.parametrize("layout", [0, 1])
@pytest.mark.parametrize("nvec", [1, 2, 3, 5, 10])
def test_curlcurl_pillbox_bit_exact(mx, ctx, orc, layout, nvec):
    A, op, ref, got, _, _ = _apply_case(mx, ctx, orc, orc.pillbox(24), "curlCurl", nvec, layout)
    assert np.array_equal(ref, got), rel_err(got, ref)
    st = A.stats()
    assert st["rows"] == op.nrows and st["nnz"] == op.nnz
    if layout == 0:
        assert st["dict_rows"] > 0.5 * op.nrows
    else:
        assert st["dict_rows"] == 0


@pytest.mark.parametrize("name", ["curlE", "curlB", "divB", "gradPsi", "vecLapl", "scaLapl", "mRhs", "gradDiv"])
def test_every_operator_on_the_path(mx, ctx, orc, name):
    """Rectangular (div/grad/curl) and assembled operators used by MxMagWaveOp::Apply (MxMagWaveOp.cpp:863-929)."""
    _, op, ref, got, _, _ = _apply_case(mx, ctx, orc, orc.pillbox(16), name, 2, None)
    assert np.array_equal(ref, got), rel_err(got, ref)


def test_vacuum32_config_c1(mx, ctx, orc):
    """BASELINE config C1: vacuum 32^3, n_B = 98304, nnz = 1277952."""
    A, op, ref, got, _, _ = _apply_case(mx, ctx, orc, orc.vacuum(32), "curlCurl", 4, None)
    assert op.nrows == 98304 and op.nnz == 1277952
    assert np.array_equal(ref, got)
    assert A.stats()["patterns"] <= 64


@pytest.mark.parametrize("layout", [0, 1])
def test_complex_bloch_matches_reference_kform_bitwise(mx, ctx, orc, layout):
    """Complex path (phase shifts -> complex entries, MxGridField.cpp:145-190). The reference stores the
    real 2N K form (MxCrsMatrix.cpp:145-170); the GPU kernel reproduces that summation order."""
    sim = orc.vacuum(12, phase_shifts=(0.4, -1.3, 2.2))
    A, op, ref, got, x, _ = _apply_case(mx, ctx, orc, sim, "curlCurl", 3, layout)
    assert op.is_complex
    assert rel_err(got, ref) < 1e-14                       # vs native complex arithmetic
    K = op.kform()
    xh = x.to_host()
    for j in range(3):
        yk = K.apply(np.ascontiguousarray(xh[:, j]).view(np.float64)).view(np.complex128)
        assert np.array_equal(yk, got[:, j])               # vs the reference's K-form order: bit-exact


def test_apply_axpby_and_aliasing_guard(mx, ctx, orc):
    sim = orc.pillbox(16)
    A, op, rmap, cmap = gpu_matrix(mx, ctx, sim, "vecLapl")
    x = mx.MxMultiVector(cmap, 3)
    y = mx.MxMultiVector(rmap, 3)
    x.random(5)
    y.random(6)
    y0 = y.to_host()
    A.apply_axpby(-1.0, x, 1.0, y)                        # residual r = b - A x (MxGeoMultigridPrec.cpp:312-314)
    ref = y0 - op.apply(x.to_host())
    assert rel_err(y.to_host(), ref) < 1e-14
    A.apply_axpby(2.5, x, 0.0, y)
    assert rel_err(y.to_host(), 2.5 * op.apply(x.to_host())) < 1e-15
    with pytest.raises(mx.MxError):
        A.apply(x, x)
    with pytest.raises(mx.MxError):
        A.apply(x, mx.MxMultiVector(rmap, 2))


def test_insert_row_values_path_sums_duplicates(mx, ctx):
    """insertRowValues + fillComplete (MxCrsMatrix.cpp:122-143,325-342): global ids, duplicates summed,
    explicit zeros kept, unsorted input accepted."""
    gids = np.array([3, 4, 9, 10, 20], dtype=np.int64)
    m = mx.MxMap(ctx, 32, gids)
    A = mx.MxCrsMatrix(m)
    A.insertRowValues(3, [4, 3, 4], [1.0, 2.0, 0.5])
    A.insertRowValues(9, [20, 3], [-1.0, 4.0])
    A.insertRowValues(10, [10], [0.0])
    A.insertRowValues(20, [9, 10, 3], [1.0, 1.0, 1.0])
    A.fillComplete(m, m)
    x = mx.MxMultiVector(m, 1)
    y = mx.MxMultiVector(m, 1)
    xv = np.array([1.0, 2.0, 3.0, 4.0, 5.0])
    x.from_host(xv)
    A.apply(x, y)
    np.testing.assert_array_equal(y.to_host()[:, 0], [2.0 * 1 + 1.5 * 2, 0.0, -5.0 + 4.0, 0.0, 3.0 + 4.0 + 1.0])
    assert A.stats()["nnz"] == 8
    B = mx.MxCrsMatrix(m)
    B.insertRowValues(3, [5], [1.0])                      # column not in the domain map
    with pytest.raises(mx.MxError):
        B.fillComplete(m, m)


def test_full_size_properties_vacuum(mx, ctx, orc):
    """Size-independent properties at a large size (no oracle apply needed): symmetry
    x.(A y) == y.(A x), gradient null space A (grad psi) = 0, linearity."""
    sim = orc.vacuum(96)
    A, op, rmap, _ = gpu_matrix(mx, ctx, sim, "curlCurl")
    G, gop, _, pmap = gpu_matrix(mx, ctx, sim, "gradPsi")
    x = mx.MxMultiVector(rmap, 2)
    y = mx.MxMultiVector(rmap, 2)
    ax = mx.MxMultiVector(rmap, 2)
    ay = mx.MxMultiVector(rmap, 2)
    x.random(1)
    y.random(2)
    A.apply(x, ax)
    A.apply(y, ay)
    lhs, rhs = ay.dot(x), ax.dot(y)
    np.testing.assert_allclose(lhs, rhs, rtol=1e-11)
    psi = mx.MxMultiVector(pmap, 2)
    psi.random(3)
    G.apply(psi, x)
    A.apply(x, ax)
    assert ax.norm2().max() <= 1e-9 * x.norm2().max() * 96 ** 2
    # linearity: A(2x - 3y) = 2Ax - 3Ay
    x.random(1)
    z = mx.MxMultiVector(rmap, 2)
    z.MvAddMv(2.0, x, -3.0, y)
    az = mx.MxMultiVector(rmap, 2)
    A.apply(z, az)
    A.apply(x, ax)
    az.MvAddMv(1.0, az, -2.0, ax)
    az.MvAddMv(1.0, az, 3.0, ay)
    assert az.norm2().max() <= 1e-12 * ay.norm2().max()


@pytest.mark.parametrize("mode", ["1", "3", "auto"])
@pytest.mark.parametrize("name,nvec", [("curlCurl", 1), ("curlCurl", 3), ("vecLapl", 6), ("scaLapl", 2), ("curlE", 1)])
def test_component_interleaved_dictionary_kernel_bit_exact(mx, ctx, orc, monkeypatch, mode, name, nvec):
    """MXG_SPMV_ILV (default auto): the dictionary kernel with warps covering 32 cells of one field component (rows r, r+3, ...).
    A different thread -> row assignment only; results stay bit-identical for every operator, also those whose rows
    do not come in triples (scaLapl) and row counts that are not multiples of the 96-row tile."""
    monkeypatch.setenv("MXG_SPMV_ILV", mode)
    _, op, ref, got, _, _ = _apply_case(mx, ctx, orc, orc.pillbox(20), name, nvec, 0)
    assert np.array_equal(ref, got), rel_err(got, ref)


@pytest.mark.parametrize("is_complex", [False, True])
def test_host_buffer_batch_apply(mx, ctx, orc, is_complex):
    """mxg_crs_apply_host_batch: y_host[i] = A x_host[i] with uploads / applies / downloads pipelined over two device
    slots; every item bit-identical to the oracle, with pinned and with pageable host buffers, for odd batch sizes."""
    sim = orc.vacuum(10, phase_shifts=(0.3, -0.2, 0.5)) if is_complex else orc.pillbox(16)
    A, op, rmap, cmap = gpu_matrix(mx, ctx, sim, "curlCurl")
    dt = np.complex128 if is_complex else np.float64
    n = op.nrows
    rng = np.random.default_rng(3)
    count = 7
    xs, ys = [], []
    for i in range(count):
        xa = mx.pinned_array((n, 1), dt) if i % 2 == 0 else np.empty((n, 1), dtype=dt)
        xa[:, 0] = rng.uniform(-1, 1, n) + (1j * rng.uniform(-1, 1, n) if is_complex else 0)
        xs.append(xa)
        ys.append(mx.pinned_array((n, 1), dt) if i % 3 == 0 else np.empty((n, 1), dtype=dt))
    A.apply_host_batch([a[:, 0] for a in xs], [a[:, 0] for a in ys])
    x = mx.MxMultiVector(cmap, 1, is_complex)
    y = mx.MxMultiVector(rmap, 1, is_complex)
    for i in range(count):
        x.from_host(xs[i])
        A.apply(x, y)
        assert np.array_equal(ys[i], y.to_host()), i
        if not is_complex:
            assert np.array_equal(ys[i], op.apply(xs[i])), i
    A.apply_host_batch([], [])


def test_literal_reference_operator_r13(mx, ctx, orc):
    """DESIGN.md R13: read literally, MxYeeFitEField::getCompFactor (MxYeeFitEField.cpp:90-98) drops curlE's wrap-around
    entries on a periodic upper boundary (MxGridField.cpp:64-74). The oracle can generate that operator too
    (literal_upper_periodic_e); the GPU apply must be bit-exact on it as on the default one -- parity is with whatever
    operator the host hands over."""
    lit, dflt = orc.vacuum(12, literal=True), orc.vacuum(12)
    _, op_l, ref_l, got_l, _, _ = _apply_case(mx, ctx, orc, lit, "curlCurl", 3, None)
    _, op_d, ref_d, got_d, _, _ = _apply_case(mx, ctx, orc, dflt, "curlCurl", 3, None)
    assert op_l.nnz < op_d.nnz                      # the literal operator lost its wrap-around couplings
    assert np.array_equal(ref_l, got_l) and np.array_equal(ref_d, got_d)
    assert not np.array_equal(got_l, got_d)


@pytest.mark.parametrize("name,size", [("curlCurl", 48), ("vecLapl", 40), ("scaLapl", 40)])
def test_windowed_kernel_equals_gather_kernel(mx, ctx, orc, name, size, monkeypatch):
    """The windowed dictionary kernel (x windows staged in shared memory by 1-D TMA, mxg_spmm_win.cuh) against the gather
    kernels (MXG_SPMV_WIN=0) and the oracle, on grids large enough for many tiles; block applies and the fused epilogue."""
    sim = orc.pillbox(size)
    monkeypatch.setenv("MXG_SPMV_WIN", "1")
    monkeypatch.setenv("MXG_WIN_MAXVEC", "128")          # default: windowed kernel for single vectors only
    Aw, op, rmap, cmap = gpu_matrix(mx, ctx, sim, name)
    monkeypatch.setenv("MXG_SPMV_WIN", "0")
    Ag, _, _, _ = gpu_matrix(mx, ctx, sim, name)
    for nvec in (1, 3, 8):
        x = mx.MxMultiVector(cmap, nvec)
        yw = mx.MxMultiVector(rmap, nvec)
        yg = mx.MxMultiVector(rmap, nvec)
        x.random(99 + nvec)
        Aw.apply(x, yw)
        Ag.apply(x, yg)
        ref = op.apply(x.to_host())
        assert np.array_equal(yg.to_host(), ref)
        assert np.array_equal(yw.to_host(), ref), (name, nvec, rel_err(yw.to_host(), ref))
        yw.random(5)
        yg.assign(yw)
        Aw.apply_axpby(-1.0, x, 1.0, yw)
        Ag.apply_axpby(-1.0, x, 1.0, yg)
        assert np.array_equal(yw.to_host(), yg.to_host())

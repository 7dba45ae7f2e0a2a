"""The CUDA multigrid preconditioner (maxwell_b200/csrc/mxg_gmg.cu) against its float64 restatement (tests/gmg_reference.py).

The reference runs with the GPU's own lambda_max, so the two differ by rounding only (about 1e-15 relative); every bound here is
1e-12, and a wrong coefficient, degree, level or projection moves the result by 1e-3 or more. Covered: 1 to 4 levels, Chebyshev
degrees 1 to 3, one and two cycles, full multigrid, the singular scalar hierarchy with remove_const_field, complex Bloch levels,
right-hand sides masked by the face fractions, calls narrower and wider than the work vectors, the operator-application count,
symmetry and positivity of the V-cycle, and the Jacobi preconditioner (the inverse diagonal every smoother uses)."""
import numpy as np
import pytest
import scipy.sparse as sp

import gmg_reference as G
from conftest import gpu_matrix

pytestmark = pytest.mark.gpu

TOL = 1e-12
BLOCH = (0.7, -0.4, 1.1)


class Hier:
    """One oracle hierarchy, uploaded: GPU level operators and transfers, and the oracle matrices for the reference."""

    def __init__(self, mx, ctx, orc, sims, name, field):
        self.sims, self.field, self.is_complex = sims, field, sims[0].is_complex
        self.ops, self.R, self.P, self.gids = G.oracle_hierarchy(orc, sims, name, field)
        self.maps = [mx.MxMap(ctx, s.num_global(field), g) for s, g in zip(sims, self.gids)]

        def up(m, rm, cm):
            rowptr, col, val = m.arrays()
            return mx.MxCrsMatrix.from_csr(rm, cm, rowptr, m.maps()[1][col], val)
        self.gops = [up(op, m, m) for op, m in zip(self.ops, self.maps)]
        self.gR = [up(r, self.maps[l + 1], self.maps[l]) for l, r in enumerate(self.R)]
        self.gP = [up(p, self.maps[l], self.maps[l + 1]) for l, p in enumerate(self.P)]

    def prec(self, mx, ctx, nlev, **kw):
        return mx.MxGeoMultigridPrec(ctx, self.gops[:nlev], self.gR[:nlev - 1], self.gP[:nlev - 1], **kw)

    def reference(self, prec, nlev, **kw):
        lam = [prec.info(l)["lambda_max"] for l in range(nlev)]
        return G.from_oracle(self.ops[:nlev], self.R[:nlev - 1], self.P[:nlev - 1], self.gids[:nlev], lambda_max=lam, **kw)

    def rhs(self, seed, ncols):
        """ncols hashed random columns; the second half is zero where the fine level's fraction is 0."""
        b = G.random_columns(seed, self.gids[0], ncols, self.is_complex)
        b[:, ncols // 2:] *= (self.sims[0].fracs(self.field) > 0)[:, None]
        return b


@pytest.fixture(scope="module")
def hiers(mx, ctx, orc):
    return {
        "vec": Hier(mx, ctx, orc, [orc.pillbox(n) for n in (32, 16, 8, 4)], "vecLapl", "bfield"),
        "sca": Hier(mx, ctx, orc, [orc.pillbox(n) for n in (32, 16, 8)], "scaLapl", "psifield"),
        "bloch": Hier(mx, ctx, orc, [orc.vacuum(n, phase_shifts=BLOCH) for n in (16, 8)], "vecLapl", "bfield"),
    }


def _apply(mx, h, prec, b):
    B = mx.MxMultiVector(h.maps[0], b.shape[1], h.is_complex)
    B.from_host(b)
    X = B.Clone(b.shape[1])
    prec.ApplyInverse(B, X)
    return X.to_host()


@pytest.mark.parametrize("hier", ["vec", "sca", "bloch"])
def test_lambda_max_is_the_restated_power_iteration(mx, ctx, hiers, hier):
    h = hiers[hier]
    prec = h.prec(mx, ctx, len(h.ops))
    for l, op in enumerate(h.ops):
        A = G.local_csr(op, h.gids[l], h.gids[l])
        want = G.power_lambda_max(A, G.inv_diag(A), h.gids[l], l)
        got = prec.info(l)["lambda_max"]
        assert abs(got - want) <= TOL * want, (l, got, want)


# (hierarchy, levels, preconditioner parameters); the V-cycles among them are also checked for symmetry
VCYCLES = [
    ("vec", 1, dict(smoother_sweeps=2)),
    ("vec", 2, dict(smoother_sweeps=2)),
    ("vec", 3, dict(smoother_sweeps=2)),
    ("vec", 4, dict(smoother_sweeps=2)),
    ("vec", 3, dict(smoother_sweeps=1)),
    ("vec", 3, dict(smoother_sweeps=3)),
    ("vec", 3, dict(smoother_sweeps=2, cycles=2)),
    ("sca", 3, dict(smoother_sweeps=2, remove_const_field=True)),
    ("sca", 2, dict(smoother_sweeps=1, remove_const_field=True)),
    ("bloch", 2, dict(smoother_sweeps=2)),
]
FMG = [
    ("vec", 3, dict(smoother_sweeps=2, full_multigrid=True)),
    ("vec", 4, dict(smoother_sweeps=2, cycles=2, full_multigrid=True)),
    ("sca", 3, dict(smoother_sweeps=2, full_multigrid=True, remove_const_field=True)),
    ("bloch", 2, dict(smoother_sweeps=2, full_multigrid=True)),
]


def _id(case):
    hier, nlev, kw = case
    return "%s-%dl-" % (hier, nlev) + "-".join("%s%s" % (k, int(v)) for k, v in sorted(kw.items()))


@pytest.mark.parametrize("case", VCYCLES + FMG, ids=_id)
def test_apply_inverse_equals_the_reference(mx, ctx, hiers, case):
    hier, nlev, kw = case
    h = hiers[hier]
    prec = h.prec(mx, ctx, nlev, **kw)
    ref = h.reference(prec, nlev, **kw)
    b = h.rhs(101, 4)
    count0 = prec.info(0)["spmm_count"]
    got = _apply(mx, h, prec, b)
    want = ref.apply(b)
    err = G.column_errors(got, want)
    assert np.all(err < TOL), err
    assert prec.info(0)["spmm_count"] - count0 == ref.count


@pytest.mark.parametrize("case", VCYCLES, ids=_id)
def test_vcycle_is_symmetric_and_positive(mx, ctx, hiers, case):
    """b2^H M^-1 b1 = conj(b1^H M^-1 b2) and b^H M^-1 b > 0: what block CG (scalar hierarchy) and LOBPCG assume of M^-1."""
    hier, nlev, kw = case
    h = hiers[hier]
    b = h.rhs(202, 4)
    x = _apply(mx, h, h.prec(mx, ctx, nlev, **kw), b)
    for i, j in ((0, 1), (2, 3), (0, 3)):
        asym, qi, qj = G.asymmetry(b[:, i], x[:, i], b[:, j], x[:, j])
        assert asym <= TOL, (i, j, asym)
        assert qi > 0 and qj > 0


@pytest.mark.parametrize("hier,kw", [("vec", dict(smoother_sweeps=2)), ("sca", dict(smoother_sweeps=2, remove_const_field=True)),
                                     ("vec", dict(smoother_sweeps=2, full_multigrid=True))], ids=["vec", "sca-rcf", "vec-fmg"])
def test_call_shapes_and_views(mx, ctx, hiers, hier, kw):
    """One preconditioner applied to 3, 1, 2 and then 5 columns: views narrower than its work vectors, then freshly allocated
    (uninitialised) work vectors. x is a non-contiguous view of a NaN-filled block: the result must not depend on what x held,
    the other columns must stay untouched, and b must come back bit for bit."""
    h = hiers[hier]
    nlev = len(h.sims) if hier == "sca" else 3
    prec = h.prec(mx, ctx, nlev, **kw)
    ref = h.reference(prec, nlev, **kw)
    for seed, nc in ((1, 3), (2, 1), (3, 2), (4, 5)):
        b = h.rhs(seed, nc)
        B = mx.MxMultiVector(h.maps[0], nc, h.is_complex)
        B.from_host(b)
        before = B.to_host()
        Xall = mx.MxMultiVector(h.maps[0], 2 * nc + 1, h.is_complex)
        Xall.MvInit(np.nan)
        cols = list(range(1, 2 * nc + 1, 2))
        X = Xall.CloneViewNonConst(cols)
        prec.ApplyInverse(B, X)
        assert np.array_equal(B.to_host(), before), "ApplyInverse wrote to b"
        xall = Xall.to_host()
        others = np.setdiff1d(np.arange(2 * nc + 1), cols)
        assert np.all(np.isnan(xall[:, others])), "ApplyInverse wrote outside the columns of x"
        err = G.column_errors(xall[:, cols], ref.apply(b))
        assert np.all(err < TOL), (nc, err)


def _jacobi_of_ones(mx, A, rmap, is_complex):
    x = mx.MxMultiVector(rmap, 1, is_complex)
    x.MvInit(1.0)
    y = mx.MxMultiVector(rmap, 1, is_complex)
    y.MvInit(np.nan)
    assert mx.load_library().mxg_crs_jacobi(A.h, x.h, y.h) == 0, mx.load_library().mxg_last_error().decode()
    return y.to_host()[:, 0]


def _assert_inverse_diagonal(got, Acsr):
    want = G.inv_diag(Acsr)
    assert np.array_equal(got.real, want.real) and np.array_equal(got.imag, want.imag), \
        "%d of %d entries differ" % (np.count_nonzero(got != want), len(want))


@pytest.mark.parametrize("case,name", [("pillbox", "vecLapl"), ("pillbox", "scaLapl"), ("bloch", "vecLapl"), ("bloch-pec", "curlCurl")])
def test_jacobi_is_the_inverse_diagonal_of_an_uploaded_operator(mx, ctx, orc, case, name):
    sim = {"pillbox": lambda: orc.pillbox(16), "bloch": lambda: orc.vacuum(8, phase_shifts=BLOCH),
           "bloch-pec": lambda: orc.Sim(12, origin=(-0.5,) * 3, size=(1.0,) * 3, phase_shifts=BLOCH,
                                        pec=orc.Shape.sphere(0.45, (0, 0, 0)))}[case]()
    A, op, rmap, _ = gpu_matrix(mx, ctx, sim, name)
    rg, cg = op.maps()
    _assert_inverse_diagonal(_jacobi_of_ones(mx, A, rmap, op.is_complex), G.local_csr(op, rg, rg))


@pytest.mark.parametrize("case,name", [("pillbox", "vecLapl"), ("pillbox", "scaLapl"), ("bloch-pec", "curlCurl")])
def test_jacobi_is_the_inverse_diagonal_of_a_device_assembled_operator(mx, ctx, case, name):
    from maxwell_b200 import assembly as asm
    if case == "pillbox":
        sim = asm.example_sim(ctx, "pillbox", 16)
    else:
        sim = asm.gpu_sim(ctx, 12, origin=(-0.5,) * 3, size=(1.0,) * 3, phase_shifts=BLOCH)
        sim.set_pec_shape(asm.gpu_api().sphere(0.45, (0, 0, 0)))
        sim.setup()
    field = "psifield" if name == "scaLapl" else "bfield"
    d = sim.op(name)
    rmap = asm.make_map(sim, field)
    A = asm.to_crs(d, rmap, rmap)
    rowptr, col, val = d.arrays()
    Acsr = sp.csr_matrix((val, col, rowptr), shape=(d.nrows, d.ncols))
    _assert_inverse_diagonal(_jacobi_of_ones(mx, A, rmap, d.is_complex), Acsr)

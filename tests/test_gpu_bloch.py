"""Phase-consistent multigrid on Bloch-periodic problems on the device (DESIGN.md GMG-bloch, include/mxasm.h: MXG_INTERP_BLOCH).

  * The device's Bloch transfers (whole, row windows, restriction windows) equal the oracle's bit for bit on the cases
    tests/test_asm_bloch_replay.py replays on the CPU.
  * The CUDA V-cycle on a device-assembled hierarchy with these transfers equals tests/gmg_reference.py to 1e-12 per
    column, and as a stationary iteration it takes the residual below 1e-6 within 30 cycles.
    Both on the periodic vacuum box and on the sapphire photonic crystal of example/phc-sapph-r0.37.py.
  * The projected complex eigensolve (Maxwell modes at k != 0) with Bloch transfers in both hierarchies, and a scalar
    hierarchy that does not remove the constant field (it is no null vector when a phase is non-zero), on the periodic
    vacuum box against its analytic transverse spectrum. (The sapphire crystal's curl-curl is not Hermitian -- the 9-point
    anisotropic inverse permittivity of MxYeeFitInvEps is not symmetric, by about 4 % of its largest entry -- so the
    Hermitian block solver does not converge on it with either transfer; DESIGN.md section 5.)
"""
import numpy as np
import pytest
import scipy.sparse as sp

import gmg_reference as G
from test_asm_bloch_replay import BLOCH_CASES, check_bloch_transfers

pytestmark = pytest.mark.gpu

PHI = (0.7, -0.4, 1.1)
PHC_PHI = (2.0, 1.1, 0.4)          # bench.py's k-point of example/phc-sapph-r0.37.py
TOL = 1e-12


class DeviceAPI:
    """The device assembly API with the simulations bound to one context (the shape of the replay API the checks take)."""

    def __init__(self, ctx):
        from maxwell_b200 import assembly as asm
        self.api, self.ctx = asm.gpu_api(), ctx

    def __getattr__(self, name):
        return getattr(self.api, name)

    def sim(self, _ctx, n, **kw):
        s = self.api.sim(self.ctx.h, n, **kw)
        s.ctx = self.ctx
        return s


@pytest.mark.parametrize("case", sorted(BLOCH_CASES) + ["phc-sapphire"])
def test_device_bloch_transfers_match_the_oracle_bit_for_bit(ctx, case):
    check_bloch_transfers(DeviceAPI(ctx), case)


def _host_csr(d):
    rowptr, col, val = d.arrays()
    return sp.csr_matrix((val, col, rowptr), shape=(d.nrows, d.ncols))


def _problem(ctx, make, sizes):
    from maxwell_b200 import assembly as asm
    sims = [make(n) for n in sizes]
    ep = asm.EigenProblem(ctx, sims, is_complex=True, bloch_transfers=True)
    return sims, ep


def _vacuum(ctx, n):
    from maxwell_b200 import assembly as asm
    return asm.gpu_sim(ctx, n, origin=(0.0,) * 3, size=(1.0,) * 3, phase_shifts=PHI).setup()


@pytest.mark.parametrize("case,name", [("vacuum", "vecLapl"), ("vacuum", "scaLapl"), ("phc", "vecLapl"), ("phc", "scaLapl")])
def test_bloch_vcycle_equals_the_reference_and_converges(mx, ctx, case, name):
    """vacuum: levels 32 / 16 / 8 at phases (0.7, -0.4, 1.1); phc: the sapphire crystal at 24 / 12 / 6, phases (2.0, 1.1, 0.4)."""
    from maxwell_b200 import assembly as asm
    field = "bfield" if name == "vecLapl" else "psifield"
    if case == "vacuum":
        sizes, make = (32, 16, 8), lambda n: _vacuum(ctx, n)
    else:
        sizes, make = (24, 12, 6), lambda n: asm.example_sim(ctx, "phc", n, phase_shifts=PHC_PHI)
    sims, ep = _problem(ctx, make, sizes)
    ops, R, P = (ep.vops, ep.Rb, ep.Pb) if name == "vecLapl" else (ep.sops, ep.Rp, ep.Pp)
    maps = ep.bmaps if name == "vecLapl" else ep.pmaps
    prec = mx.MxGeoMultigridPrec(ctx, ops, R, P, smoother_sweeps=2)
    # the reference on the same device-assembled matrices, with the GPU's lambda_max
    A = [_host_csr(s.op(name, True)) for s in sims]
    Ph = [_host_csr(sims[l].interpolator_from(sims[l + 1], field, True, bloch=True)) for l in range(len(sims) - 1)]
    Rh = [(p.conj().T / 8.0).tocsr() for p in Ph]
    gids = [s.map(field) for s in sims]
    ref = G.Multigrid(A, Rh, Ph, gids, lambda_max=[prec.info(l)["lambda_max"] for l in range(len(sims))], smoother_sweeps=2)
    b = G.random_columns(101, gids[0], 4, True)
    B = mx.MxMultiVector(maps[0], 4, True)
    B.from_host(b)
    X = B.Clone(4)
    prec.ApplyInverse(B, X)
    err = G.column_errors(X.to_host(), ref.apply(b))
    assert np.all(err < TOL), err
    # stationary iteration x <- x + M^-1 (b - A x)
    x = mx.MxMultiVector(maps[0], 4, True)
    r, e = B.CloneCopy(), B.Clone(4)
    r0 = r.norm2()
    hist = []
    for _ in range(30):
        prec.ApplyInverse(r, e)
        x.MvAddMv(1.0, x, 1.0, e)
        r.assign(B)
        ops[0].apply_axpby(-1.0, x, 1.0, r)
        hist.append((r.norm2() / r0).max())
        if hist[-1] < 1e-6:
            break
    print("%s %s: %d cycles to %.2e (rate %.3f)" % (case, name, len(hist), hist[-1], hist[-1] ** (1.0 / len(hist))))
    assert hist[-1] < 1e-6, hist


def _solve(mx, ctx, ep, nev, block=16):
    from maxwell_b200 import assembly as asm
    prec = mx.MxGeoMultigridPrec(ctx, ep.vops, ep.Rb, ep.Pb, smoother_sweeps=2)
    rcf = asm.scalar_laplacian_has_constant_null_vector(ep.sims[0])
    assert not rcf
    sprec = mx.MxGeoMultigridPrec(ctx, ep.sops, ep.Rp, ep.Pp, smoother_sweeps=2, remove_const_field=rcf)
    s = mx.MxSolver(ctx, ep.vops[0], m_diag=ep.m_diag, prec=prec, nev=nev, block_size=block, tol=1e-9, max_iters=300,
                    projection={"divB": ep.divB, "gradPsi": ep.gradPsi, "scaLapl": ep.sops[0], "sca_prec": sprec})
    ev = s.solve()
    assert s.converged == nev, (s.converged, s.residuals)
    res, div = s.check(ep.divB, A=ep.curlCurl)
    print("iterations %d, V-cycles %d, projection block-CG iterations %d, re-projections %d"
          % (s.iterations, s.apply_prec, s.proj_cg_iters, s.reprojections))
    assert np.all(res[:nev] < 1e-6), res[:nev]
    assert np.all(div[:nev] < 1e-6), div[:nev]
    return np.asarray(ev), s


def test_projected_bloch_vacuum_modes_are_the_analytic_transverse_spectrum(mx, ctx):
    """Periodic unit box with Bloch phases: the Yee curl-curl on divergence-free fields has the eigenvalues
    sum_d (2 N sin((2 pi m_d + phi_d) / (2 N)))^2, twice each (two transverse polarisations per wave vector)."""
    N, nev = 16, 10
    _, ep = _problem(ctx, lambda n: _vacuum(ctx, n), (N, N // 2, N // 4))
    ev, s = _solve(mx, ctx, ep, nev)
    m = np.arange(-3, 4)
    M = np.stack(np.meshgrid(m, m, m, indexing="ij"), axis=-1).reshape(-1, 3)
    lam = np.sum((2.0 * N * np.sin((2.0 * np.pi * M + np.array(PHI)) / (2.0 * N))) ** 2, axis=1)
    ref = np.sort(np.repeat(lam, 2))[:nev]
    np.testing.assert_allclose(ev, ref, rtol=1e-9)
    assert s.iterations < 80, s.iterations

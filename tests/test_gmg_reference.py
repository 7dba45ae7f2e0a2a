"""The float64 multigrid reference (tests/gmg_reference.py) against textbook forms, without a GPU: the Chebyshev smoother is the
residual polynomial T_d((theta - t) / h) / T_d(theta / h) of D^-1 A, the V-cycles are symmetric (Hermitian) operators, and the
power-iteration estimate puts the smoothing interval's upper end above the spectrum of D^-1 A. tests/test_gpu_gmg.py then pins
the CUDA preconditioner to this reference."""
import numpy as np
import pytest
import scipy.sparse as sp
import scipy.sparse.linalg as sla

import gmg_reference as G


def _spd(n=7, seed=0):
    """2-D Laplacian on an n x n grid plus a random positive diagonal: SPD with a non-constant diagonal."""
    t = sp.diags([-np.ones(n - 1), 2.0 * np.ones(n), -np.ones(n - 1)], [-1, 0, 1])
    A = sp.kronsum(t, t) + sp.diags(np.random.default_rng(seed).uniform(0.1, 3.0, n * n))
    return sp.csr_matrix(A)


@pytest.mark.parametrize("degree", [1, 2, 3, 30])
def test_chebyshev_smoother_is_the_residual_polynomial(degree):
    A = _spd()
    d = A.diagonal()
    s = sp.diags(1.0 / np.sqrt(d))
    lam, Q = np.linalg.eigh((s @ A @ s).toarray())                           # D^-1/2 A D^-1/2 = Q diag(lam) Q^T
    rho = lam.max()
    ratio = 30.0
    mg = G.Multigrid([A], [], [], [None], lambda_max=[rho], smoother_sweeps=degree, eig_ratio=ratio)
    # zero-start smoothing x = S b on the columns of A: I - S A is the error propagator
    E = np.eye(A.shape[0]) - mg.apply(A.toarray())
    alpha, beta = rho / ratio, 1.1 * rho
    theta, h = 0.5 * (beta + alpha), 0.5 * (beta - alpha)
    Td = np.polynomial.chebyshev.Chebyshev.basis(degree)
    r = Td((theta - lam) / h) / Td(theta / h)
    want = (Q * r) @ Q.T * np.sqrt(np.outer(1.0 / d, d))                     # D^-1/2 Q r(lam) Q^T D^1/2
    assert np.abs(E - want).max() < 1e-12
    assert mg.count == degree - 1                                            # the zero start skips one operator application


@pytest.fixture(scope="module")
def hierarchies(orc):
    out = {}
    pill = [orc.pillbox(n) for n in (32, 16, 8)]
    out["vec"] = G.oracle_hierarchy(orc, pill, "vecLapl", "bfield")
    out["sca"] = G.oracle_hierarchy(orc, pill, "scaLapl", "psifield")
    bloch = [orc.vacuum(n, phase_shifts=(0.7, -0.4, 1.1)) for n in (16, 8)]
    out["bloch"] = G.oracle_hierarchy(orc, bloch, "vecLapl", "bfield")
    return out


def _levels(h, n):
    ops, R, P, gids = h
    return ops[:n], R[:n - 1], P[:n - 1], gids[:n]


SYMMETRIC_CYCLES = [
    ("vec", 3, dict(smoother_sweeps=2)),
    ("vec", 3, dict(smoother_sweeps=3)),
    ("vec", 3, dict(smoother_sweeps=2, cycles=2)),
    ("bloch", 2, dict(smoother_sweeps=2)),
    ("sca", 3, dict(smoother_sweeps=2)),
    ("sca", 3, dict(smoother_sweeps=2, remove_const_field=True)),
    ("sca", 2, dict(smoother_sweeps=2, remove_const_field=True)),
]


@pytest.mark.parametrize("hier,nlev,kw", SYMMETRIC_CYCLES)
def test_restated_vcycle_is_symmetric_and_positive(hierarchies, hier, nlev, kw):
    """b2^H M^-1 b1 = conj(b1^H M^-1 b2): the preconditioner CG and LOBPCG need. With remove_const_field this holds only
    because the fine residual is projected before the restriction, as well as the restricted right-hand side and the
    correction (without it the scalar cycle's asymmetry is about 1e-3)."""
    ops, R, P, gids = _levels(hierarchies[hier], nlev)
    mg = G.from_oracle(ops, R, P, gids, **kw)
    b = G.random_columns(17, gids[0], 2, ops[0].is_complex)
    x = mg.apply(b)
    asym, q1, q2 = G.asymmetry(b[:, 0], x[:, 0], b[:, 1], x[:, 1])
    assert asym < 1e-14, asym
    assert q1 > 0 and q2 > 0


@pytest.mark.parametrize("hier", ["vec", "sca"])
def test_chebyshev_interval_covers_the_spectrum(hierarchies, hier):
    ops, R, P, gids = hierarchies[hier]
    mg = G.from_oracle(ops, R, P, gids)
    for l, A in enumerate(mg.A):
        rho = abs(sla.eigs(sp.diags(mg.dinv[l]) @ A, k=1, which="LM", tol=1e-10, return_eigenvectors=False)[0])
        # 30 power steps land 2-3 % low; the 10 % margin of the interval covers it
        assert rho <= 1.1 * mg.lambda_max[l] < 1.1 * rho, (l, rho, mg.lambda_max[l])

"""Phase-consistent grid transfers (DESIGN.md GMG-bloch) on the float64 multigrid restatement (tests/gmg_reference.py), CPU only.

A Bloch-periodic field satisfies u(x + L e_d) = e^{i phi_d} u(x). The plain trilinear interpolator takes the coarse value
of a stencil cell beyond a periodic face from the cell it wraps to, without that factor, so near the wrap it does not map
a coarse Bloch field onto the fine one, and the V-cycle built on it diverges as a stationary iteration. With the factor:
  * P applied to a sampled coarse Bloch plane wave e^{i k.x}, k_d = (2 pi m_d + phi_d) / L_d, equals the fine samples to
    the trilinear error bound h^2 / 8 sum_d k_d^2 on every row, the wrap rows included (the plain P misses it there by
    far, and so would the opposite sign of the factor);
  * x <- x + M^-1 (b - A x) contracts by at most 0.65 per cycle over 20 V(2,2) cycles on vacuum and sapphire photonic
    crystal hierarchies, for the vector and the scalar Laplacian;
  * the V-cycle stays Hermitian (to 1e-14).
"""
import numpy as np
import pytest

import gmg_reference as G
import bloch_oracle as BO
from oracle import oracle as orc

PHI = (0.7, -0.4, 1.1)
PHC_PHI = (2.0, 1.1, 0.4)          # bench.py's k-point of example/phc-sapph-r0.37.py


def positions(sim, field, size, origin):
    """Coordinates of every DOF of a field's map (cell-relative Yee positions as the assembly places them)."""
    n = np.array(sim.n)
    d = np.array(size) / n
    gids = sim.map(field)
    ncomp = 1 if field == "psifield" else 3
    comp, node = gids % ncomp, gids // ncomp
    cell = np.stack([node // ((n[1] + 1) * (n[2] + 1)), (node // (n[2] + 1)) % (n[1] + 1), node % (n[2] + 1)], axis=1)
    x = np.array(origin) + cell * d
    if field == "psifield":
        return x + 0.5 * d
    xi = np.array([[0, 0.5, 0.5], [0.5, 0, 0.5], [0.5, 0.5, 0]]) * d          # B components: face centres
    return x + xi[comp]


@pytest.mark.parametrize("field", ["bfield", "psifield"])
@pytest.mark.parametrize("m", [(0, 0, 0), (1, 0, -1)])
def test_bloch_transfer_interpolates_a_bloch_plane_wave(field, m):
    size, origin = (1.0, 1.2, 0.8), (0.0, 0.0, 0.0)
    fine = orc.Sim((16, 12, 8), origin=origin, size=size, phase_shifts=PHI)
    coarse = orc.Sim((8, 6, 4), origin=origin, size=size, phase_shifts=PHI)
    k = (2.0 * np.pi * np.array(m) + np.array(PHI)) / np.array(size)
    wave = lambda s: np.exp(1j * positions(s, field, size, origin) @ k)
    uc, uf = wave(coarse), wave(fine)
    hc = np.array(size) / np.array(coarse.n)
    bound = np.sum(hc ** 2 * k ** 2) / 8.0 * (1.0 + 1e-9) + 1e-13
    P = BO.interpolator(coarse, fine, field=field, is_complex=True, bloch=True)
    P0 = orc.interpolator(coarse, fine, field=field, is_complex=True)
    err = np.abs(P.apply(uc) - uf)
    err0 = np.abs(P0.apply(uc) - uf)
    assert err.max() <= bound, (err.max(), bound)
    # the wrap rows (where the factor makes a difference) are where the plain transfer fails
    wrap = np.abs(P.scipy() - P0.scipy()).sum(axis=1).A1 > 0
    assert wrap.sum() > 0
    assert np.all(err0[~wrap] <= bound)
    far = 20.0 if m == (0, 0, 0) else 1.5          # the bound is loose for the shorter wave of m != 0
    assert err0[wrap].max() > far * bound, (err0[wrap].max(), bound)
    # the opposite sign of the factor is as wrong as no factor
    Pc = BO.interpolator(orc.Sim((8, 6, 4), origin=origin, size=size, phase_shifts=tuple(-p for p in PHI)),
                          orc.Sim((16, 12, 8), origin=origin, size=size, phase_shifts=tuple(-p for p in PHI)),
                          field=field, is_complex=True, bloch=True)
    assert np.abs(np.conj(Pc.apply(np.conj(uc))) - uf)[wrap].max() <= bound      # conj of the -phi transfer is this one
    assert np.abs(Pc.apply(uc) - uf)[wrap].max() > far * bound


def bloch_hierarchy(make, sizes, name, field):
    sims = [make(n) for n in sizes]
    ops = [s.op(name) for s in sims]
    gids = [op.maps()[0] for op in ops]
    P = [BO.interpolator(sims[l + 1], sims[l], field=field, is_complex=True, bloch=True) for l in range(len(sims) - 1)]
    R = [p.transpose(scale=1.0 / 8.0) for p in P]
    return G.from_oracle(ops, R, P, gids, smoother_sweeps=2), ops[0], gids[0]


HIERARCHIES = {
    "vacuum-vec-16-8": (lambda n: orc.vacuum(n, phase_shifts=PHI), (16, 8), "vecLapl", "bfield"),
    "vacuum-vec-32-16-8": (lambda n: orc.vacuum(n, phase_shifts=PHI), (32, 16, 8), "vecLapl", "bfield"),
    "vacuum-sca-32-16-8": (lambda n: orc.vacuum(n, phase_shifts=PHI), (32, 16, 8), "scaLapl", "psifield"),
    "phc-vec-24-12": (lambda n: orc.phc_sapphire(n, phase_shifts=PHC_PHI), (24, 12), "vecLapl", "bfield"),
    "phc-sca-24-12": (lambda n: orc.phc_sapphire(n, phase_shifts=PHC_PHI), (24, 12), "scaLapl", "psifield"),
}


@pytest.fixture(scope="module")
def hierarchies():
    return {}


def hierarchy(cache, key):
    if key not in cache:
        cache[key] = bloch_hierarchy(*HIERARCHIES[key])
    return cache[key]


@pytest.mark.parametrize("key", sorted(HIERARCHIES))
def test_stationary_vcycle_contracts_on_bloch_levels(hierarchies, key):
    mg, _, gids = hierarchy(hierarchies, key)
    A = mg.A[0]
    b = G.random_columns(31, gids, 2, True)
    x = np.zeros_like(b)
    r0 = np.linalg.norm(b, axis=0)
    hist = [np.ones(2)]
    for _ in range(20):
        x = x + mg.apply(b - A @ x)
        hist.append(np.linalg.norm(b - A @ x, axis=0) / r0)
    hist = np.array(hist)
    rate = hist[-1] ** (1.0 / 20.0)
    late = (hist[-1] / hist[10]) ** (1.0 / 10.0)
    assert np.all(rate <= 0.65) and np.all(late <= 0.65), (key, rate, late, hist[:, 0])


@pytest.mark.parametrize("key", ["vacuum-vec-32-16-8", "phc-sca-24-12"])
def test_bloch_vcycle_is_hermitian(hierarchies, key):
    mg, _, gids = hierarchy(hierarchies, key)
    b = G.random_columns(77, gids, 2, True)
    x = mg.apply(b)
    asym, q1, q2 = G.asymmetry(b[:, 0], x[:, 0], b[:, 1], x[:, 1])
    assert asym <= 1e-14 and q1 > 0 and q2 > 0, (asym, q1, q2)

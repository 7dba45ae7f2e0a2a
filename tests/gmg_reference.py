"""Plain float64 restatement of the multigrid preconditioner of maxwell_b200/csrc/mxg_gmg.cu (numpy / scipy, one process).

It states what the CUDA cycle must compute, so that a kernel change (a fused smoother, an FP32 cycle) can be measured against a
tolerance instead of a contraction rate. Rounding makes the CUDA result differ from this one by about 1e-15 relative; any error
of a coefficient, a degree, a level or a projection is 1e-3 or larger.

Restated here, each next to the routine it follows:
  inv_diag            k_lb_inv_diag / lbInverse (mxg_spmv.cu): dInvDiag of every operator
  power_lambda_max    estimateLambdaMax: 30 steps of u <- D^-1 A (u / |u|) from a hashed random start, lambda = |u|
  Multigrid.smooth    smooth: Chebyshev on D^-1 A over [lambda / ratio, 1.1 lambda], the Ifpack recurrence
  Multigrid.vcycle    vcycle, with "remove const field" on the fine residual, the restricted right-hand side and the correction
  Multigrid.apply     applyImpl: `cycles` V-cycles, or full multigrid
  Multigrid.count     operator applications, as info(0)["spmm_count"] counts them
Operators are scipy CSR matrices in the order of each level's map; vectors are (rows, columns) arrays.
"""
import numpy as np
import scipy.sparse as sp

from maxwell_b200 import hash_uniform


def local_csr(mat, row_gids, col_gids):
    """An oracle Matrix as scipy CSR with rows in the order of row_gids and columns in the order of col_gids."""
    rowptr, col, val = mat.arrays()
    rg, cg = mat.maps()
    assert np.array_equal(rg, row_gids), "rows of the operator are not in the order of the level map"
    order = np.argsort(col_gids)
    pos = order[np.searchsorted(col_gids, cg, sorter=order)]
    assert np.array_equal(col_gids[pos], cg), "operator columns outside the level map"
    return sp.csr_matrix((val, pos[col], rowptr), shape=(len(row_gids), len(col_gids)))


def oracle_hierarchy(orc, sims, name="vecLapl", field="bfield"):
    """Level operators `name` on the oracle simulations `sims` (fine to coarse), trilinear prolongations P[l] (level l+1 -> l)
    and restrictions R[l] = P[l]^H / 8, as oracle matrices, plus each level's GIDs (the order of its map)."""
    cx = sims[0].is_complex
    ops = [s.op(name) for s in sims]
    gids = [op.maps()[0] for op in ops]
    P = [orc.interpolator(sims[l + 1], sims[l], field=field, is_complex=cx) for l in range(len(sims) - 1)]
    R = [p.transpose(scale=1.0 / 8.0) for p in P]
    return ops, R, P, gids


def inv_diag(A):
    """1 / diag(A), 0 where the diagonal is 0 or absent. Complex: (re / m2, -im / m2) with m2 = re*re + im*im, every product
    and the sum rounded on its own, as lbInverse computes it (so the result can be compared bit for bit)."""
    d = A.diagonal()
    nz = d != 0
    out = np.zeros_like(d)
    if np.iscomplexobj(d):
        re, im = d.real[nz], d.imag[nz]
        m2 = re * re + im * im
        out.real[nz] = re / m2
        out.imag[nz] = -im / m2
    else:
        out[nz] = 1.0 / d[nz]
    return out


def random_columns(seed, gids, ncols, is_complex):
    """MvRandom (mxg_mv_random) of a fresh block: column j from hash_uniform(seed, gid, j), imaginary part from part 1."""
    x = np.empty((len(gids), ncols), dtype=np.complex128 if is_complex else np.float64)
    for j in range(ncols):
        x[:, j] = hash_uniform(seed, gids, j, 0)
        if is_complex:
            x[:, j] += 1j * hash_uniform(seed, gids, j, 1)
    return x


def power_lambda_max(A, dinv, gids, level, iters=30):
    """estimateLambdaMax: lambda_max(D^-1 A) by `iters` power steps from MvRandom(0x5eed + level)."""
    u = random_columns(0x5eed + level, gids, 1, np.iscomplexobj(dinv))[:, 0]
    lam = 1.0
    for _ in range(iters):
        nrm = np.linalg.norm(u)
        if nrm == 0.0:
            break
        u = dinv * (A @ (u * (1.0 / nrm)))
        lam = np.linalg.norm(u)
    return lam


def remove_const_field(x):
    """mxg_mv_remove_const_field: subtract each column's mean."""
    return x - x.sum(axis=0) / x.shape[0]


class Multigrid:
    """The V-cycle / full-multigrid preconditioner of mxg_gmg on scipy operators (fine to coarse), with the parameters of
    mxg_gmg_default_params. lambda_max: one value per level (default: the restated power iteration)."""

    def __init__(self, ops, R, P, gids, lambda_max=None, smoother_sweeps=2, cycles=1, eig_ratio=30.0, coarse_degree=30,
                 coarse_eig_ratio=1000.0, full_multigrid=False, power_iterations=30, remove_const_field=False):
        self.A, self.R, self.P = list(ops), list(R), list(P)
        self.nlevels = len(self.A)
        self.dinv = [inv_diag(A) for A in self.A]
        if lambda_max is None:
            lambda_max = [power_lambda_max(A, d, g, l, power_iterations) for l, (A, d, g) in enumerate(zip(self.A, self.dinv, gids))]
        self.lambda_max = [float(v) for v in lambda_max]
        self.degree, self.cycles, self.ratio = int(smoother_sweeps), int(cycles), float(eig_ratio)
        self.coarse_degree, self.coarse_ratio = int(coarse_degree), float(coarse_eig_ratio)
        self.fmg, self.rcf = bool(full_multigrid), bool(remove_const_field)
        self.count = 0

    def _applyA(self, l, x):
        self.count += 1
        return self.A[l] @ x

    def smooth(self, l, x, b, degree, ratio, zero_start):
        """Chebyshev smoother of `degree` on D^-1 A; zero_start: x is taken as 0 (and not read)."""
        if degree <= 0:
            return x
        lmax = self.lambda_max[l]
        alpha, beta = lmax / ratio, 1.1 * lmax
        delta, theta = 2.0 / (beta - alpha), 0.5 * (beta + alpha)
        s1 = theta * delta
        d = self.dinv[l][:, None]
        if zero_start:
            w = (1.0 / theta) * (d * b)
            x = w
        else:
            w = (1.0 / theta) * (d * (b - self._applyA(l, x)))
            x = x + w
        rhok = 1.0 / s1
        for _ in range(1, degree):
            v = self._applyA(l, x)
            rhokp1 = 1.0 / (2.0 * s1 - rhok)
            c1, c2 = rhokp1 * rhok, 2.0 * rhokp1 * delta
            rhok = rhokp1
            w = c1 * w + c2 * (d * (b - v))
            x = x + w
        return x

    def vcycle(self, l, x, b, zero_start):
        if l == self.nlevels - 1:
            one = self.nlevels == 1
            return self.smooth(l, x, b, self.degree if one else self.coarse_degree, self.ratio if one else self.coarse_ratio, zero_start)
        x = self.smooth(l, x, b, self.degree, self.ratio, zero_start)
        r = b - self._applyA(l, x)
        if self.rcf:
            r = remove_const_field(r)
        self.count += 1
        bc = self.R[l] @ r
        if self.rcf:
            bc = remove_const_field(bc)
        xc = self.vcycle(l + 1, None, bc, True)
        self.count += 1
        e = self.P[l] @ xc
        if self.rcf:
            e = remove_const_field(e)
        x = x + e
        return self.smooth(l, x, b, self.degree, self.ratio, False)

    def apply(self, b):
        """ApplyInverse: x = M^-1 b for a (rows, columns) block b."""
        b = np.asarray(b)
        if not self.fmg or self.nlevels == 1:
            x = self.vcycle(0, None, b, True)
            for _ in range(1, self.cycles):
                x = self.vcycle(0, x, b, False)
            return x
        bl = [b]
        for l in range(1, self.nlevels):
            self.count += 1
            bc = self.R[l - 1] @ bl[l - 1]
            bl.append(remove_const_field(bc) if self.rcf else bc)
        last = self.nlevels - 1
        x = self.smooth(last, None, bl[last], self.coarse_degree, self.coarse_ratio, True)
        for l in range(last - 1, -1, -1):
            self.count += 1
            x = self.P[l] @ x
            if self.rcf:
                x = remove_const_field(x)
            for _ in range(self.cycles):
                x = self.vcycle(l, x, bl[l], False)
        return x


def from_oracle(ops, R, P, gids, **params):
    """Multigrid on oracle matrices as oracle_hierarchy returns them."""
    n = len(ops)
    A = [local_csr(ops[l], gids[l], gids[l]) for l in range(n)]
    Rs = [local_csr(R[l], gids[l + 1], gids[l]) for l in range(n - 1)]
    Ps = [local_csr(P[l], gids[l], gids[l + 1]) for l in range(n - 1)]
    return Multigrid(A, Rs, Ps, gids, **params)


def asymmetry(b1, x1, b2, x2):
    """|b2^H M^-1 b1 - conj(b1^H M^-1 b2)| / sqrt(b1^H M^-1 b1 * b2^H M^-1 b2) for x_i = M^-1 b_i; 0 for a symmetric
    (Hermitian) M^-1. Also returns the two quadratic forms b_i^H M^-1 b_i (real parts)."""
    q1, q2 = np.vdot(b1, x1).real, np.vdot(b2, x2).real
    return abs(np.vdot(b2, x1) - np.conj(np.vdot(b1, x2))) / np.sqrt(abs(q1 * q2)), q1, q2


def column_errors(got, ref):
    """Relative 2-norm error of every column."""
    return np.linalg.norm(got - ref, axis=0) / np.linalg.norm(ref, axis=0)

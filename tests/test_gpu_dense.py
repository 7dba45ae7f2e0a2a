"""Tall-skinny block products (MvTransMv: k_gram_mma, complex k_trans_mv; MvTimesMatAddMv: k_update_mma, k_times_mat) and
the column reductions (k_dot_partial, k_sum_partial) against exact references.

Most data are small integers, the scalars dyadic and the B matrices integer, so every partial sum is an integer below 2^53:
the float64 numpy reference is then exact in any summation order and the kernels must match it bit for bit. A dropped row, a
stale chunk, a wrong column slot or a wrong partial slice is off by at least 1. A few full-mantissa cases hold the kernels to
the worst-case FP64 bound against a long-double reference, which no float32 path can meet.

Which instantiation and launch grid each shape reaches is restated in tests/dense_plan.py; the first test checks on this
device's SM count that the sweep reaches every instantiation and at least 3 ring iterations per CTA."""
import numpy as np
import pytest

import dense_plan as plan

pytestmark = pytest.mark.gpu

ROWS = 1 << 17          # row block of the host-side references


@pytest.fixture(scope="module")
def sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def test_sweep_premise_on_this_device(sms):
    got = plan.premise(sms)
    assert got["min_gram_iters"] >= 3 and got["min_update_iters"] >= 3


# ---- helpers ------------------------------------------------------------------------------------------------------------
def _map(mx, ctx, n):
    return mx.MxMap(ctx, 2 * n + 5, np.arange(n, dtype=np.int64) * 2 + 1)


def _ints(rng, n, c, cplx=False, lim=8):
    """(n, c) column-major integers in [-lim, lim] (complex: integer real and imaginary parts), compactly typed."""
    if cplx:
        re = rng.integers(-lim, lim + 1, size=(c, n), dtype=np.int8).T
        im = rng.integers(-lim, lim + 1, size=(c, n), dtype=np.int8).T
        return np.asfortranarray(re + 1j * im.astype(np.complex64))
    return rng.integers(-lim, lim + 1, size=(c, n), dtype=np.int8).T


def _upload(mv, h, cols=None):
    """host columns h[:, j] -> mv column cols[j] (16 columns at a time, to keep the float64 copy small)"""
    cols = list(range(h.shape[1])) if cols is None else list(cols)
    for j0 in range(0, len(cols), 16):
        j1 = min(j0 + 16, len(cols))
        mv.CloneView(cols[j0:j1]).from_host(h[:, j0:j1].astype(mv.dtype))


def _gram_ref(Ah, Xh, dtype):
    """Ah^H Xh, row block by row block (exact on integer data)"""
    G = np.zeros((Ah.shape[1], Xh.shape[1]), dtype=dtype)
    for r0 in range(0, Ah.shape[0], ROWS):
        G += Ah[r0:r0 + ROWS].astype(dtype).conj().T @ Xh[r0:r0 + ROWS].astype(dtype)
    return G


def _cols(rng, total, k, style):
    """column list of a view: contiguous, reversed, a random reordered subset, or every other column"""
    if style == 0:
        s = (total - k) // 2
        return list(range(s, s + k))
    if style == 1:
        return list(range(k - 1, -1, -1))
    if style == 3 and 2 * k <= total:
        return list(range(1, 2 * k, 2))
    return [int(c) for c in rng.permutation(total)[:k]]


def _first_bad(got, want):
    bad = np.argwhere(~(got == want))
    return "%d of %d entries differ, first (row, col): %s" % (len(bad), got.size, bad[:4].tolist())


def _check_update(got, Ah, ca, B, alpha, beta, Y0, what):
    """got == alpha * Ah[:, ca] B + beta * Y0 exactly, row block by row block"""
    assert got.shape == (Ah.shape[0], B.shape[1]), what
    for r0 in range(0, Ah.shape[0], ROWS):
        want = alpha * (Ah[r0:r0 + ROWS][:, ca].astype(got.dtype) @ B)
        if beta != 0:
            want = want + beta * Y0[r0:r0 + ROWS].astype(got.dtype)
        blk = got[r0:r0 + ROWS]
        assert np.array_equal(blk, want), what + (r0, _first_bad(blk, want))


SCALARS = [(-0.5, 2.0), (0.75, 0.5), (2.0, -1.0), (1.0, 0.0), (-1.0, 0.25)]
CSCALARS = [(0.5 - 0.25j, 0.75 + 0.5j), (-2.0 + 1.0j, 0.0), (1.0, -0.5j)]


# ---- real sweep at 2^20 + 35 rows ---------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def pool(mx, ctx):
    """one integer A and one integer X of 128 columns each; every shape below is a view of them"""
    n = plan.SWEEP_N
    rng = np.random.default_rng(20)
    m = _map(mx, ctx, n)
    Ah, Xh = _ints(rng, n, plan.MAX_COLS), _ints(rng, n, plan.MAX_COLS)
    A, X = mx.MxMultiVector(m, plan.MAX_COLS), mx.MxMultiVector(m, plan.MAX_COLS)
    _upload(A, Ah)
    _upload(X, Xh)
    return {"n": n, "map": m, "A": A, "X": X, "Ah": Ah, "Xh": Xh,
            "AX": _gram_ref(Ah, Xh, np.float64), "AA": _gram_ref(Ah, Ah, np.float64)}


@pytest.mark.parametrize("k,b", plan.GRAM_SHAPES)
def test_gram_sweep(pool, k, b):
    rng = np.random.default_rng(1000 * k + b)
    ca, cx = _cols(rng, plan.MAX_COLS, k, (k + b) % 4), _cols(rng, plan.MAX_COLS, b, (k + 2 * b + 1) % 4)
    alpha = SCALARS[(k + b) % len(SCALARS)][0]
    G = pool["X"].CloneView(cx).MvTransMv(alpha, pool["A"].CloneView(ca))
    want = alpha * pool["AX"][np.ix_(ca, cx)]
    assert np.array_equal(G, want), ("gram", k, b, _first_bad(G, want))


@pytest.mark.parametrize("k,b", [(1, 1), (17, 17), (48, 48), (33, 96), (128, 128)])
def test_gram_of_overlapping_views(pool, k, b):
    """A and X are views of the same block (the Rayleigh-Ritz Grams of one basis): shared and permuted columns"""
    rng = np.random.default_rng(k + 7 * b)
    ca, cx = _cols(rng, plan.MAX_COLS, k, 2), _cols(rng, plan.MAX_COLS, b, 2)
    G = pool["A"].CloneView(cx).MvTransMv(1.0, pool["A"].CloneView(ca))
    assert np.array_equal(G, pool["AA"][np.ix_(ca, cx)]), ("gram of one block", k, b)
    if k == b == plan.MAX_COLS:
        assert np.array_equal(pool["A"].MvTransMv(-0.5, pool["A"]), -0.5 * pool["AA"])


@pytest.mark.parametrize("k,b", plan.UPDATE_SHAPES)
def test_update_sweep(mx, pool, k, b):
    rng = np.random.default_rng(3000 * k + b)
    ca = _cols(rng, plan.MAX_COLS, k, (k + b) % 4)
    alpha, beta = SCALARS[(k + 3 * b) % len(SCALARS)]
    B = rng.integers(-4, 5, size=(k, b)).astype(np.float64)
    Y = mx.MxMultiVector(pool["map"], b)
    yc = [int(c) for c in rng.permutation(b)]                    # Y is written through a reordered view
    Yv = Y.CloneView(yc)
    Y0 = _ints(rng, pool["n"], b)
    _upload(Yv, Y0)
    Yv.MvTimesMatAddMv(alpha, pool["A"].CloneView(ca), B, beta)
    _check_update(Yv.to_host(), pool["Ah"], ca, B, alpha, beta, Y0, ("update", k, b, alpha, beta))


@pytest.mark.parametrize("k", plan.IN_PLACE_K)
def test_in_place_right_multiplication(mx, pool, k):
    """base(:, dst) = base(:, src) C with dst a reordered subset of src (MxSolver.hpp rightMul), one pass over the block"""
    rng = np.random.default_rng(k)
    W = mx.MxMultiVector(pool["map"], plan.UPDATE_MAX_K)
    Wh = pool["Ah"][:, :plan.UPDATE_MAX_K]
    _upload(W, Wh)
    src = [int(c) for c in rng.permutation(plan.UPDATE_MAX_K)[:k]]
    nd = min(k, plan.UPDATE_PASS_COLS)
    dst = src[::-1][:nd] if k != plan.UPDATE_MAX_K else [int(c) for c in rng.permutation(src)[:nd]]
    C = rng.integers(-3, 4, size=(k, nd)).astype(np.float64)
    W.CloneView(dst).MvTimesMatAddMv(1.0, W.CloneView(src), C, 0.0)
    got = W.to_host()
    rest = [c for c in range(plan.UPDATE_MAX_K) if c not in dst]
    assert np.array_equal(got[:, rest], Wh[:, rest].astype(np.float64)), ("in place: a column outside dst changed", k)
    _check_update(np.asfortranarray(got[:, dst]), Wh, src, C, 1.0, 0.0, None, ("in place", k))


# ---- complex sweep ------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def cpool(mx, ctx):
    n = plan.CPLX_N
    rng = np.random.default_rng(21)
    m = _map(mx, ctx, n)
    Ah, Xh = _ints(rng, n, 64, True), _ints(rng, n, 64, True)
    A, X = mx.MxMultiVector(m, 64, True), mx.MxMultiVector(m, 64, True)
    _upload(A, Ah)
    _upload(X, Xh)
    return {"n": n, "map": m, "A": A, "X": X, "Ah": Ah, "Xh": Xh, "AX": _gram_ref(Ah, Xh, np.complex128)}


@pytest.mark.parametrize("k,b", plan.CPLX_GRAM_SHAPES)
def test_complex_gram_sweep(cpool, k, b):
    rng = np.random.default_rng(5000 * k + b)
    ca, cx = _cols(rng, 64, k, (k + b) % 4), _cols(rng, 64, b, (k + b + 2) % 4)
    alpha = CSCALARS[(k + b) % len(CSCALARS)][0]
    G = cpool["X"].CloneView(cx).MvTransMv(alpha, cpool["A"].CloneView(ca))
    want = alpha * cpool["AX"][np.ix_(ca, cx)]
    assert np.array_equal(G, want), ("complex gram", k, b, _first_bad(G, want))


@pytest.mark.parametrize("k,b", plan.CPLX_UPDATE_SHAPES)
def test_complex_update_sweep(mx, cpool, k, b):
    rng = np.random.default_rng(7000 * k + b)
    ca = _cols(rng, 64, k, (k + b) % 4)
    alpha, beta = CSCALARS[(k + b) % len(CSCALARS)]
    B = rng.integers(-4, 5, size=(k, b)) + 1j * rng.integers(-4, 5, size=(k, b))
    Y = mx.MxMultiVector(cpool["map"], b, True)
    Yv = Y.CloneView([int(c) for c in rng.permutation(b)])
    Y0 = _ints(rng, cpool["n"], b, True)
    _upload(Yv, Y0)
    Yv.MvTimesMatAddMv(alpha, cpool["A"].CloneView(ca), B, beta)
    _check_update(Yv.to_host(), cpool["Ah"], ca, B, alpha, beta, Y0, ("complex update", k, b))


# ---- row-count edges ----------------------------------------------------------------------------------------------------
EDGE = ["0", "1", "15", "16", "63", "64", "65", "127", "128", "chunks=ctas", "chunks=ctas+1"]


@pytest.mark.parametrize("which", EDGE)
def test_row_count_edges(mx, ctx, sms, which):
    """An empty map (the Gram is zero, the update a no-op), a tail chunk shorter than / equal to / one past 64 rows (an odd
    tail makes the bulk copy read one padded element), and chunk counts equal to and one above the CTA count."""
    n = plan.edge_rows(sms)[EDGE.index(which)]
    rng = np.random.default_rng(n)
    m = _map(mx, ctx, n)
    Ah, Xh = _ints(rng, n, 72), _ints(rng, n, 96)
    A, X = mx.MxMultiVector(m, 72), mx.MxMultiVector(m, 96)
    _upload(A, Ah)
    _upload(X, Xh)
    for k, b in [(1, 1), (5, 17), (33, 2), (48, 48), (64, 96)]:
        ca, cx = _cols(rng, 72, k, 2), _cols(rng, 96, b, 2)
        G = X.CloneView(cx).MvTransMv(-0.5, A.CloneView(ca))
        want = -0.5 * _gram_ref(Ah[:, ca], Xh[:, cx], np.float64)
        assert np.array_equal(G, want), ("gram", n, k, b, _first_bad(G, want))
    for k, b in [(3, 17), (64, 48), (64, 49), (65, 20)]:
        ca = _cols(rng, 72, k, 2)
        B = rng.integers(-4, 5, size=(k, b)).astype(np.float64)
        Y = mx.MxMultiVector(m, b)
        Y0 = _ints(rng, n, b)
        _upload(Y, Y0)
        Y.MvTimesMatAddMv(0.75, A.CloneView(ca), B, 2.0)
        _check_update(Y.to_host(), Ah, ca, B, 0.75, 2.0, Y0, ("update", n, k, b))
    Ac, Xc = _ints(rng, n, 5, True), _ints(rng, n, 7, True)
    A, X = mx.MxMultiVector(m, 5, True), mx.MxMultiVector(m, 7, True)
    _upload(A, Ac)
    _upload(X, Xc)
    G = X.MvTransMv(0.5 - 0.25j, A)
    assert np.array_equal(G, (0.5 - 0.25j) * _gram_ref(Ac, Xc, np.complex128)), ("complex gram", n)
    B = rng.integers(-4, 5, size=(5, 7)) + 1j * rng.integers(-4, 5, size=(5, 7))
    X.MvTimesMatAddMv(1.0 + 1.0j, A, B, -0.5)
    _check_update(X.to_host(), Ac, list(range(5)), B, 1.0 + 1.0j, -0.5, Xc, ("complex update", n))
    x = A.CloneView([0, 3])
    sq = (Ac[:, [0, 3]].real.astype(np.int64) ** 2 + Ac[:, [0, 3]].imag.astype(np.int64) ** 2).sum(axis=0)
    assert np.array_equal(x.norm2(), np.sqrt(sq.astype(np.float64))), ("complex norm2", n)


# ---- reductions ---------------------------------------------------------------------------------------------------------
def _reduction_rows(sms):
    out = [(1 << 20, 1), (1 << 20, 5)]
    for nc in (1, 5):
        e = plan.unroll_edge_rows(nc, sms, 1 << 20)
        out += [(e, nc), (e + 1, nc)]
    return out


@pytest.mark.parametrize("cplx", [False, True])
def test_dot_norm_remove_const_field(mx, ctx, sms, cplx):
    """dot and norm2 are exact on integer data at rows that end exactly on, and one past, the two-way unrolled stride of
    k_dot_partial; remove_const_field is exact when the row count is a power of two (1/count is exact)."""
    for n, nc in _reduction_rows(sms):
        rng = np.random.default_rng(n + nc)
        m = _map(mx, ctx, n)
        Ah, Bh = _ints(rng, n, nc, cplx), _ints(rng, n, nc, cplx)
        A, B = mx.MxMultiVector(m, nc, cplx), mx.MxMultiVector(m, nc, cplx)
        _upload(A, Ah)
        _upload(B, Bh)
        if cplx:
            a, b = Ah.astype(np.complex128), Bh.astype(np.complex128)
            ar, ai, br, bi = (v.astype(np.int64) for v in (a.real, a.imag, b.real, b.imag))
            want = (ar * br + ai * bi).sum(axis=0) + 1j * (ar * bi - ai * br).sum(axis=0)
            sq = (ar * ar + ai * ai).sum(axis=0)
        else:
            a64, b64 = Ah.astype(np.int64), Bh.astype(np.int64)
            want = (a64 * b64).sum(axis=0).astype(np.float64)
            sq = (a64 * a64).sum(axis=0)
        assert np.array_equal(B.dot(A), want), ("dot", n, nc, cplx)
        assert np.array_equal(A.norm2(), np.sqrt(sq.astype(np.float64))), ("norm2", n, nc, cplx)
        A.remove_const_field()
        got = A.to_host()
        s = Ah.astype(np.complex128 if cplx else np.int64).sum(axis=0)
        want = Ah.astype(got.dtype) - (s.astype(got.dtype) * (1.0 / n))[None, :]
        if n & (n - 1) == 0:
            assert np.array_equal(got, want), ("remove_const_field", n, nc, cplx)
        else:  # the kernel may fuse the multiply into the subtraction: one rounding apart at most
            tol = 2 * np.finfo(np.float64).eps * (np.abs(Ah.astype(got.dtype)) + np.abs(s / n)[None, :])
            assert np.all(np.abs(got - want) <= tol), ("remove_const_field", n, nc, cplx)


# ---- B with a leading dimension above k ---------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def mid(mx, ctx):
    n = 40009
    rng = np.random.default_rng(40009)
    m = _map(mx, ctx, n)
    Ah, Ach = _ints(rng, n, 72), _ints(rng, n, 16, True)
    A, Ac = mx.MxMultiVector(m, 72), mx.MxMultiVector(m, 16, True)
    _upload(A, Ah)
    _upload(Ac, Ach)
    return {"n": n, "map": m, "A": A, "Ah": Ah, "Ac": Ac, "Ach": Ach}


@pytest.mark.parametrize("cplx", [False, True])
def test_ldb_above_k(mid, cplx):
    """MvTransMv writes only the first k rows of an (ldb x b) B, MvTimesMatAddMv reads only the first k rows of one (the
    TMA-staged update for k <= 64, the parameter-block update above, and the complex one)"""
    A, Ah = (mid["Ac"], mid["Ach"]) if cplx else (mid["A"], mid["Ah"])
    dt = np.complex128 if cplx else np.float64
    for k, b, ldb in ([(5, 3, 9), (13, 3, 17)] if cplx else [(20, 7, 29), (48, 33, 50), (65, 7, 70)]):
        rng = np.random.default_rng(k + ldb)
        ca, cx = list(range(k)), list(range(A.GetNumberVecs() - b, A.GetNumberVecs()))
        sentinel = np.full((ldb, b), -777.25 + (3j if cplx else 0), dtype=dt, order="F")
        out = sentinel.copy(order="F")
        got = A.CloneView(cx).MvTransMv(2.0, A.CloneView(ca), ldb=ldb, out=out)
        assert got is out and np.array_equal(out[k:], sentinel[k:]), ("rows k..ldb of B were written", k, b, ldb)
        assert np.array_equal(out[:k], 2.0 * _gram_ref(Ah[:, ca], Ah[:, cx], dt)), ("gram with ldb", k, b, ldb)
        Bf = np.full((ldb, b), np.nan, dtype=dt, order="F")
        Bf[:k] = rng.integers(-4, 5, size=(k, b)) + (1j * rng.integers(-4, 5, size=(k, b)) if cplx else 0)
        Y = A.Clone(b)
        Y.MvTimesMatAddMv(0.5, A.CloneView(ca), Bf, 0.0, ldb=ldb)
        _check_update(Y.to_host(), Ah, ca, Bf[:k], 0.5, 0.0, None, ("update with ldb", k, b, ldb))


@pytest.mark.parametrize("k,b,cplx", [(30, 20, False), (64, 49, False), (65, 17, False), (5, 7, True)])
def test_nan_filled_y_with_zero_beta(mid, k, b, cplx):
    """beta = 0 overwrites Y: NaNs already there must not leak into the result"""
    A, Ah = (mid["Ac"], mid["Ach"]) if cplx else (mid["A"], mid["Ah"])
    rng = np.random.default_rng(k * 31 + b)
    B = rng.integers(-4, 5, size=(k, b)) + (1j * rng.integers(-4, 5, size=(k, b)) if cplx else 0)
    Y = A.Clone(b)
    Y.MvInit(float("nan"))
    ca = _cols(rng, A.GetNumberVecs(), k, 2)
    Y.MvTimesMatAddMv(0.5, A.CloneView(ca), B, 0.0)
    _check_update(Y.to_host(), Ah, ca, np.asarray(B, dtype=Y.dtype), 0.5, 0.0, None, ("NaN-filled Y", k, b))


# ---- full-mantissa data against a long-double reference -----------------------------------------------------------------
U = 2.0 ** -53


def _gamma(m):
    return m * U / (1 - m * U)


@pytest.mark.parametrize("k,b", [(48, 32), (17, 5), (64, 49)])
def test_gram_full_mantissa(mx, ctx, k, b):
    """|G - G_ref| <= gamma_n |A|^T |X| entry by entry, for any summation order; a float32 contraction misses it by orders
    of magnitude"""
    n = 40009
    rng = np.random.default_rng(k * b)
    m = _map(mx, ctx, n)
    Ah, Xh = np.asfortranarray(rng.uniform(-1, 1, (n, k))), np.asfortranarray(rng.uniform(-1, 1, (n, b)))
    A, X = mx.MxMultiVector(m, k), mx.MxMultiVector(m, b)
    A.from_host(Ah)
    X.from_host(Xh)
    G = X.MvTransMv(1.0, A)
    ref = Ah.astype(np.longdouble).T @ Xh.astype(np.longdouble)
    bound = _gamma(n) * (np.abs(Ah).T @ np.abs(Xh))
    err = np.abs(G.astype(np.longdouble) - ref)
    assert np.all(err <= bound), ("gram", k, b, float((err / bound).max()))
    g32 = (Ah.astype(np.float32).T @ Xh.astype(np.float32)).astype(np.longdouble)
    assert np.any(np.abs(g32 - ref) > bound)                     # the bound does separate FP64 from FP32


@pytest.mark.parametrize("k,b", [(30, 17), (64, 48), (65, 20)])
def test_update_full_mantissa(mx, ctx, k, b):
    n = 40009
    rng = np.random.default_rng(k + 100 * b)
    m = _map(mx, ctx, n)
    Ah, Yh = np.asfortranarray(rng.uniform(-1, 1, (n, k))), np.asfortranarray(rng.uniform(-1, 1, (n, b)))
    B = rng.uniform(-1, 1, (k, b))
    alpha, beta = -0.7, 1.3
    A, Y = mx.MxMultiVector(m, k), mx.MxMultiVector(m, b)
    A.from_host(Ah)
    Y.from_host(Yh)
    Y.MvTimesMatAddMv(alpha, A, B, beta)
    L = np.longdouble
    ref = L(alpha) * (Ah.astype(L) @ B.astype(L)) + L(beta) * Yh.astype(L)
    bound = _gamma(k + 2) * (abs(alpha) * (np.abs(Ah) @ np.abs(B)) + abs(beta) * np.abs(Yh))
    err = np.abs(Y.to_host().astype(L) - ref)
    assert np.all(err <= bound), ("update", k, b, float((err / bound).max()))


def test_complex_full_mantissa(mx, ctx):
    n, k, b = 40009, 13, 6
    rng = np.random.default_rng(13)
    m = _map(mx, ctx, n)
    cu = lambda *s: rng.uniform(-1, 1, s) + 1j * rng.uniform(-1, 1, s)  # noqa: E731
    Ah, Xh, B = np.asfortranarray(cu(n, k)), np.asfortranarray(cu(n, b)), cu(k, b)
    A, X = mx.MxMultiVector(m, k, True), mx.MxMultiVector(m, b, True)
    A.from_host(Ah)
    X.from_host(Xh)
    G = X.MvTransMv(1.0, A)
    L = np.clongdouble
    ref = Ah.astype(L).conj().T @ Xh.astype(L)
    bound = _gamma(2 * n + 2) * (np.abs(Ah).T @ np.abs(Xh))
    for part in (np.real, np.imag):
        assert np.all(np.abs(part(G.astype(L) - ref)) <= bound), ("complex gram", part.__name__)
    X.MvTimesMatAddMv(1.0, A, B, 0.0)
    ref = Ah.astype(L) @ B.astype(L)
    bound = _gamma(2 * k + 2) * (np.abs(Ah) @ np.abs(B))
    got = X.to_host().astype(L)
    for part in (np.real, np.imag):
        assert np.all(np.abs(part(got - ref)) <= bound), ("complex update", part.__name__)

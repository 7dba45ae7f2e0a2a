"""Launch plan of the tall-skinny block products, restated from maxwell_b200/csrc/mxg_mvops.cu so that a test can say which
kernel instantiation a shape reaches and how many pipeline iterations each CTA runs, without a GPU.

Restated (line numbers of mxg_mvops.cu):
  transMvImpl   :373-437  Gram C = A^H X. Real: k_gram_mma<ri, rj> on a (gtiles, gs) grid, ri / rj from k / b (:387), gs CTAs
                          per tile capped by the chunk count (:389-394), two partial slices per CTA (:395). Complex:
                          k_trans_mv<zd, 4, 4> on a (tiles, slices) grid with a grid-stride loop over kBlock rows (:376-383).
  timesMatImpl  :440-499  Update Y = alpha A B + beta Y. Real with k <= kUpdateMaxK: one k_update_mma<RC> pass per 48
                          output columns, grid = min(chunks, 2 SMs) (:450-478). Otherwise k_times_mat<T, BT, 2>: one
                          parameter block of kMaxBParam doubles per launch group, BT columns per launch (:480-497).
  dotToScratch  :339-356  k_dot_partial on an (np, ncols) grid, two-way unrolled over a stride of np * kBlock rows.
  mxg_mv_times_mat_add_mv :747-757  in-place right-multiplication is allowed for real A with <= kUpdateMaxK columns and
                          <= 48 result columns.
In mxg_dense.cuh every CTA of k_gram_mma / k_update_mma walks the 64-row chunks blockIdx, blockIdx + gridDim, ... through
a two-stage ring: iteration it uses stage it & 1 with barrier parity (it >> 1) & 1, so three iterations are the least that
refill a consumed stage, and four reach parity 1 on both stages.
"""

K_BLOCK = 256          # kBlock
DENSE_ROWS = 64        # kDenseRows
UPDATE_MAX_K = 64      # kUpdateMaxK
MAX_B_PARAM = 1536     # kMaxBParam (doubles)
UPDATE_PASS_COLS = 48  # output columns of one k_update_mma pass
MAX_COLS = 128         # MXG_MAX_COLS


def cdiv(a, b):
    return -(-a // b)


def grid_for(sms, work, block, per_sm):
    """gridFor (mxg_internal.h)."""
    return min(max(cdiv(work, block), 1), sms * per_sm)


def gram_tile(k, b):
    """(ri, rj) of k_gram_mma: the C tile is (16 ri) x (16 rj)."""
    ri = 3 if k >= 33 else cdiv(k, 16)
    rj = 3 if b >= 33 else cdiv(b, 16)
    return ri, rj


def gram_plan(k, b, n, sms, cplx=False):
    if cplx:
        kt, bt = 4, 4
        tiles = cdiv(k, kt) * cdiv(b, bt)
        slices = max(min(cdiv(sms * 4, tiles), cdiv(n, K_BLOCK)), 1)
        return {"kernel": "k_trans_mv", "inst": (kt, bt), "grid": (tiles, slices),
                "min_iters": n // (slices * K_BLOCK), "partial_tile": k % kt != 0 or b % bt != 0}
    ri, rj = gram_tile(k, b)
    gtiles = cdiv(k, 16 * ri) * cdiv(b, 16 * rj)
    chunks = cdiv(n, DENSE_ROWS)
    gs = max(min(cdiv(sms * 2, gtiles), chunks), 1)
    # CTA y takes chunks y, y + gs, ...: the last one (y = gs - 1) gets the fewest
    return {"kernel": "k_gram_mma", "inst": (ri, rj), "grid": (gtiles, gs), "chunks": chunks, "slices": 2 * gs,
            "min_chunks_per_cta": chunks // gs, "max_chunks_per_cta": cdiv(chunks, gs)}


def update_plan(k, b, n, sms, cplx=False):
    """One entry per kernel launch."""
    if n == 0:
        return []
    if not cplx and k <= UPDATE_MAX_K:
        out = []
        chunks = cdiv(n, DENSE_ROWS)
        grid = min(chunks, 2 * sms)
        for c0 in range(0, b, UPDATE_PASS_COLS):
            cc = min(UPDATE_PASS_COLS, b - c0)
            out.append({"kernel": "k_update_mma", "inst": cdiv(cc, 16), "cols": (c0, cc), "grid": grid, "chunks": chunks,
                        "min_chunks_per_cta": chunks // grid, "k4": (k + 3) & ~3})
        return out
    w = 2 if cplx else 1
    bt = 8 if cplx else 16
    per_launch = MAX_B_PARAM // (k * w)
    if per_launch < 1:
        raise ValueError("A has too many columns for one pass")
    grid = grid_for(sms, n, K_BLOCK * 2, 4)
    out = []
    for c0 in range(0, b, per_launch):
        cc = min(per_launch, b - c0)
        for j0 in range(0, cc, bt):
            out.append({"kernel": "k_times_mat", "inst": (bt, 2), "cols": (c0 + j0, min(bt, cc - j0)), "grid": grid,
                        "min_iters": n // (grid * K_BLOCK * 2)})
    return out


def in_place_ok(k, b, cplx=False):
    return not cplx and k <= UPDATE_MAX_K and b <= UPDATE_PASS_COLS


def dot_plan(n, ncols, sms):
    """k_dot_partial: np blocks per column; the unrolled loop covers 2 * stride rows per iteration."""
    np_ = max(min(grid_for(sms, n, K_BLOCK * 8, 4), cdiv(sms * 4, ncols)), 1)
    stride = np_ * K_BLOCK
    return {"np": np_, "stride": stride, "tail": n % (2 * stride)}


def unroll_edge_rows(ncols, sms, near):
    """A row count close to `near` that ends exactly on the two-way unrolled stride of k_dot_partial (and n + 1 does not)."""
    np_ = min(sms * 4, cdiv(sms * 4, ncols))      # the block count once the rows fill 4 blocks per SM (n >= 8 np kBlock)
    n = max(round(near / (2 * K_BLOCK * np_)), 4) * 2 * K_BLOCK * np_
    assert dot_plan(n, ncols, sms)["tail"] == 0 and dot_plan(n + 1, ncols, sms)["tail"] == 1
    return n


# ---- the sweep of tests/test_gpu_dense.py ------------------------------------------------------------------------------
SWEEP_N = (1 << 20) + 35            # 16385 chunks of 64 rows: the last one holds 35 rows
SMALL = (1, 5, 16, 17, 32, 33, 48)  # every (ri, rj) of k_gram_mma, partial and full 16-column tiles
WIDE = (49, 64, 96, 128)            # several C tiles per Gram
GRAM_SHAPES = [(k, b) for k in SMALL for b in SMALL] + [(k, b) for k in WIDE for b in WIDE]
# update: RC = 1, 2, 3; k mod 4 = 0..3 (zero-padded DMMA k steps); k = 64 / 65 either side of the k_times_mat switch;
# b = 49, 96, 128 with k <= 64 (several passes through the one device copy of B); k > 64 with several parameter blocks
UPDATE_SHAPES = [(1, 1), (2, 16), (3, 17), (4, 32), (5, 33), (13, 48), (30, 7), (47, 40), (64, 48), (65, 48), (64, 49),
                 (56, 96), (61, 128), (96, 33), (128, 128)]
IN_PLACE_K = (48, 56, 64)
CPLX_N = (1 << 19) + 21
CPLX_GRAM_SHAPES = [(1, 1), (5, 7), (13, 50), (49, 3), (64, 64)]
CPLX_UPDATE_SHAPES = [(1, 1), (5, 7), (13, 70), (50, 40), (64, 64)]


def edge_rows(sms):
    """Row counts of the edge cases: empty, shorter than / equal to / one past a chunk, and chunk counts equal to and one
    above the CTA count of a one-tile Gram and of the update (2 SMs)."""
    return [0, 1, 15, 16, 63, 64, 65, 127, 128, 2 * sms * DENSE_ROWS, 2 * sms * DENSE_ROWS + 1]


def premise(sms):
    """What the sweep reaches on a device with `sms` SMs; raises AssertionError when a premise of the sweep fails."""
    gram = [gram_plan(k, b, SWEEP_N, sms) for k, b in GRAM_SHAPES]
    insts = {p["inst"] for p in gram}
    assert insts == {(ri, rj) for ri in (1, 2, 3) for rj in (1, 2, 3)}, insts
    assert min(p["min_chunks_per_cta"] for p in gram) >= 3, "a Gram CTA runs fewer than 3 ring iterations"
    assert any(p["grid"][0] > 1 for p in gram)
    upd = [(k, b, u) for k, b in UPDATE_SHAPES for u in update_plan(k, b, SWEEP_N, sms)]
    mma = [u for _, _, u in upd if u["kernel"] == "k_update_mma"]
    assert {u["inst"] for u in mma} == {1, 2, 3}
    assert min(u["min_chunks_per_cta"] for u in mma) >= 3, "an update CTA runs fewer than 3 ring iterations"
    assert {k % 4 for k, b, u in upd if u["kernel"] == "k_update_mma"} == {0, 1, 2, 3}
    assert any(k == UPDATE_MAX_K for k, b in UPDATE_SHAPES) and any(k == UPDATE_MAX_K + 1 for k, b in UPDATE_SHAPES)
    multipass = {b for k, b in UPDATE_SHAPES if k <= UPDATE_MAX_K and len(update_plan(k, b, SWEEP_N, sms)) > 1}
    assert {49, 96, 128} <= multipass, multipass
    tm = [u for _, _, u in upd if u["kernel"] == "k_times_mat"]
    assert any(u["cols"][1] < 16 for u in tm) and min(u["min_iters"] for u in tm) >= 1
    assert all(in_place_ok(k, min(k, UPDATE_PASS_COLS)) for k in IN_PLACE_K) and max(IN_PLACE_K) == UPDATE_MAX_K
    cg = [gram_plan(k, b, CPLX_N, sms, True) for k, b in CPLX_GRAM_SHAPES]
    assert any(p["partial_tile"] for p in cg) and any(k > 48 for k, _ in CPLX_GRAM_SHAPES)
    assert min(p["min_iters"] for p in cg) >= 2, "a complex Gram thread runs its grid-stride loop fewer than 2 times"
    cu = [(k, b, update_plan(k, b, CPLX_N, sms, True)) for k, b in CPLX_UPDATE_SHAPES]
    assert any(len({u["cols"][0] - u["cols"][0] % (MAX_B_PARAM // (2 * k)) for u in us}) > 1 for k, b, us in cu), \
        "no complex update needs several parameter blocks"
    assert any(u["cols"][1] < 8 for _, _, us in cu for u in us) and any(k > 48 for k, _, _ in cu)
    assert min(u["min_iters"] for _, _, us in cu for u in us) >= 1
    rows = edge_rows(sms)
    assert gram_plan(1, 1, rows[-2], sms)["grid"][1] == 2 * sms and gram_plan(1, 1, rows[-2], sms)["max_chunks_per_cta"] == 1
    assert gram_plan(1, 1, rows[-1], sms)["max_chunks_per_cta"] == 2
    assert update_plan(3, 17, rows[-1], sms)[0]["grid"] == 2 * sms
    return {"gram_insts": sorted(insts), "update_insts": sorted({u["inst"] for u in mma}),
            "min_gram_iters": min(p["min_chunks_per_cta"] for p in gram),
            "min_update_iters": min(u["min_chunks_per_cta"] for u in mma)}

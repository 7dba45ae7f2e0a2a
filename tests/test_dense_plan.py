"""CPU checks of tests/dense_plan.py: the dense-product sweep of tests/test_gpu_dense.py reaches every kernel instantiation
and the steady state of the two-stage ring on a 148-SM B200, and the constants the plan restates still match the source."""
import os
import re

import dense_plan as plan

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_sweep_premise_on_b200():
    got = plan.premise(148)
    assert got["min_gram_iters"] >= 3 and got["min_update_iters"] >= 3


def test_edge_rows_and_unroll_edges():
    for sms in (132, 148):
        rows = plan.edge_rows(sms)
        assert rows[:2] == [0, 1] and plan.gram_plan(1, 1, 0, sms)["grid"] == (1, 1)
        assert plan.update_plan(3, 17, 0, sms) == []
        for ncols in (1, 5):
            n = plan.unroll_edge_rows(ncols, sms, 1 << 20)
            assert plan.dot_plan(n, ncols, sms)["tail"] == 0 and plan.dot_plan(n + 1, ncols, sms)["tail"] == 1


def test_plan_constants_match_the_source():
    src = open(os.path.join(ROOT, "maxwell_b200", "csrc", "mxg_mvops.cu")).read()
    dense = open(os.path.join(ROOT, "maxwell_b200", "csrc", "mxg_dense.cuh")).read()
    head = open(os.path.join(ROOT, "include", "mxgpu.h")).read()
    assert re.search(r"constexpr int kBlock = %d;" % plan.K_BLOCK, src)
    assert re.search(r"constexpr int kUpdateMaxK = %d;" % plan.UPDATE_MAX_K, src)
    assert re.search(r"constexpr int kMaxBParam = %d;" % plan.MAX_B_PARAM, src)
    assert re.search(r"constexpr int kDenseRows = %d;" % plan.DENSE_ROWS, dense)
    assert re.search(r"#define MXG_MAX_COLS %d\b" % plan.MAX_COLS, head)
    # the launch choices the plan restates, as written in transMvImpl / timesMatImpl / dotToScratch
    for line in ("const int ri = k >= 33 ? 3 : (k + 15) / 16, rj = b >= 33 ? 3 : (b + 15) / 16;",
                 "int gs = (ctx->numSMs * 2 + gtiles - 1) / gtiles;",
                 "if (w == 1) slices = 2 * gs;",
                 "constexpr int KT = (w == 1) ? 8 : 4, BT = 4;",
                 "int slices = (ctx->numSMs * 4 + tiles - 1) / tiles;",
                 "for (int c0 = 0; c0 < b; c0 += 48) {",
                 "const int grid = int(std::min<int64_t>(chunks, int64_t(ctx->numSMs) * 2));",
                 "constexpr int BT = (w == 1) ? 16 : 8;",
                 "const int colsPerLaunch = kMaxBParam / (k * w);",
                 "const int grid = gridFor(ctx, Y->ld, kBlock * RT, 4);",
                 "int np = gridFor(ctx, a->ld, kBlock * 8, 4);",
                 "int cap = (ctx->numSMs * 4 + nc - 1) / nc;",
                 "const bool inPlaceOk = !A->isComplex && A->ncols <= kUpdateMaxK && Y->ncols <= 48;"):
        assert line in src, line

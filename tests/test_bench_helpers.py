"""Host-side helpers of bench.py: the algorithmic-byte formula of SURVEY.md section 8(d), the DOF-balanced x-slab
cut, the nvidia-smi clock sampler's parsing and the files of --dump-outputs. No GPU."""
import importlib.util
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
bench = importlib.util.module_from_spec(spec)
spec.loader.exec_module(bench)


def test_crs_equivalent_bytes_match_survey_figures():
    # C1 vacuum-32, one vector: 12 * 1,277,952 + 98,304 * 20 = 17.30 MB
    assert bench.crs_bytes(1277952, 98304, 1, False) == 12 * 1277952 + 98304 * 20 == 17301504
    # vacuum-256: 8.858 GB
    assert abs(bench.crs_bytes(654311424, 50331648, 1, False) / 1e9 - 8.858) < 1e-3
    # complex: 20 bytes per entry, 32 per vector element
    assert bench.crs_bytes(10, 2, 3, True) == 200 + 2 * (4 + 96)
    # block of b vectors only adds vector traffic
    assert bench.crs_bytes(100, 10, 4, False) - bench.crs_bytes(100, 10, 1, False) == 10 * 16 * 3


def test_slab_ranges_cut_on_planes_and_balance(orc):
    n = 16
    sim = orc.pillbox(n)
    gids = sim.map("bfield")
    n_global = sim.num_global("bfield")
    plane = n_global // (n + 1)
    for nranks in (1, 2, 3, 4, 8):
        cuts = bench.slab_ranges(gids, n_global, nranks, n)
        assert cuts[0] == 0 and cuts[-1] == len(gids) and len(cuts) == nranks + 1
        assert all(b >= a for a, b in zip(cuts, cuts[1:]))
        for c in cuts[1:-1]:
            # every cut falls on the first DOF of an x-plane: a rank owns whole planes (one contiguous GID range)
            assert c == len(gids) or gids[c] // plane > gids[c - 1] // plane
        sizes = np.diff(cuts)
        if nranks <= 4:
            assert sizes.max() <= 1.5 * len(gids) / nranks        # the PEC mask is uneven; the cut balances DOFs


def test_clock_sampler_summary_parses_nvidia_smi_rows():
    s = bench.ClockSampler(0)
    s.samples = [(10.0, "1965, 1965, Not Active, Not Active, Not Active, Not Active"),
                 (10.1, "1950, 1965, Not Active, Not Active, Not Active, Active"),
                 (10.2, "1965, 1965, Not Active, Not Active, Not Active, Not Active"),
                 (99.0, "300, 1965, Active, Not Active, Not Active, Not Active")]
    out = s.summary(10.0, 10.2)
    assert out["sm_mhz"] == 1965.0 and out["sm_max_mhz"] == 1965.0 and out["samples"] == 3
    assert out["reasons"] == ["sw_power_cap"]                      # the sample outside the timed window is ignored
    s.samples = []
    assert s.summary(0, 1)["samples"] == 0


def test_dump_outputs_sample_is_fixed_and_fits(tmp_path):
    """--dump-outputs: outputs of two builds are compared row for row, so the sample must not depend on the run."""
    assert np.array_equal(bench.dump_rows(1000, 16), np.arange(1000))
    n = 50_000_000                                                  # ~ pillbox-256 B-field rows
    rows = bench.dump_rows(n, 8)
    assert np.array_equal(rows, bench.dump_rows(n, 8))
    assert len(rows) * 8 <= bench.DUMP_BYTES < 64 << 20
    assert rows[0] >= 0 and rows[-1] < n and np.all(np.diff(rows) > 0)
    y = np.array([[1 + 2j], [3 - 4j]])
    bench.write_outputs(str(tmp_path / "d"), {"y": y, "ev": [2.5, 7.0]})
    got = np.load(tmp_path / "d" / "y.npy")
    assert got.dtype == np.float64 and got.shape == (2, 1, 2) and np.array_equal(got[..., 0] + 1j * got[..., 1], y)
    assert np.load(tmp_path / "d" / "ev.npy").tolist() == [2.5, 7.0]


def test_dump_outputs_slabs_concatenate_to_the_global_sample(orc):
    """Every rank dumps the sampled rows of its slab; rank 0 concatenates the pieces in rank order."""
    n = 16
    sim = orc.pillbox(n)
    gids = sim.map("bfield")
    n_global = sim.num_global("bfield")
    y = np.arange(len(gids), dtype=np.float64) * 3.0 + 1.0     # stands for the global y = A x
    rows = bench.dump_rows(len(gids), bench.DUMP_BYTES // (len(gids) // 3))
    assert 0 < len(rows) < len(gids)                           # a real sample, not every row
    for nranks in (1, 2, 3, 4):
        cuts = bench.slab_ranges(gids, n_global, nranks, n)
        pieces = [y[r0:r1][bench.slab_dump_rows(rows, r0, r1)] for r0, r1 in zip(cuts, cuts[1:])]
        assert np.array_equal(np.concatenate(pieces), y[rows])

"""Pin the CPU oracle against outputs recorded from the unmodified reference.

The fixtures in tests/golden/ were written by oracle/make_golden.py, which imports the
reference from /root/reference and calls its own methods.  If these fail the oracle is
wrong and no GPU parity claim that leans on it means anything.
"""

import hashlib

import numpy as np
import pytest

from oracle import parrm_oracle as oracle
from oracle.golden_inputs import checked_filter_edges_inputs
from pyparrm_b200 import get_example_data_paths
from pyparrm_b200.synthetic import make_recording

DIRECTIONS = ("both", "past", "future")


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def edge_mask(n_times, taps):
    """True where at least one tap is in range (outside SURVEY S2's FFT-noise zone)."""
    return oracle.in_range_tap_count(n_times, taps) > 0


def test_taps_bit_exact(golden):
    g = golden("taps")
    table, starts, taps = g["table"], g["starts"], g["taps"]
    for row, (per, phw, hw, omit, d, n, n_taps) in enumerate(table):
        mine = oracle.tap_offsets(per, phw, int(hw), int(omit), DIRECTIONS[int(d)])
        ref = taps[starts[row] : starts[row + 1]]
        if n_taps < 0:
            assert mine.shape[0] == 0
            with pytest.raises(RuntimeError, match="A suitable filter cannot be created"):
                oracle.build_filter(per, phw, int(hw), int(omit), DIRECTIONS[int(d)])
        else:
            assert np.array_equal(mine, ref), f"row {row}: {table[row]}"


def test_default_half_width(golden):
    g = golden("taps")
    for row, (per, phw, hw, omit, d, n, n_taps) in enumerate(g["table"]):
        if int(n) > 100_000:
            continue  # the scalar loop is slow; the long cases are covered by the host test
        assert oracle.default_half_width(per, phw, int(omit), int(n)) == g["default_half_width"][row]


def test_objective_matches_reference(golden):
    g = golden("objective")
    n, fs, fa = g["recording"]
    cache = {}
    for case in range(int(g["n_cases"])):
        n_chans, bw, lam, seed = g[f"case{case}_params"]
        key = (int(n_chans), int(seed))
        if key not in cache:
            data = make_recording(int(n_chans), int(n), float(fs), float(fa), seed=int(seed))
            cache[key] = oracle.standardise(data, 3.0)
        z = cache[key]
        periods, want = g[f"case{case}_periods"], g[f"case{case}_values"]
        got = oracle.objective_many(periods[::4], z, g[f"case{case}_indices"], int(bw), float(lam))
        np.testing.assert_allclose(got, want[::4], rtol=1e-12, atol=0)


def test_filter_fft_and_direct_match_reference(golden):
    g = golden("filter_edges")
    for case, x in enumerate(checked_filter_edges_inputs(g)):
        taps, hw, want = g[f"case{case}_taps"], int(g[f"case{case}_hw"]), g[f"case{case}_y"]
        filt = np.zeros(2 * hw + 1)
        filt[taps.astype(np.int64) + hw] = -1.0 / taps.shape[0]
        filt[hw] = 1
        np.testing.assert_array_equal(oracle.apply_filter_fft(x, filt), want)
        ok = edge_mask(x.shape[1], taps)
        direct = oracle.apply_filter_direct(x, taps)
        scale = max(1.0, np.abs(x).max())
        if ok.any():
            assert np.abs(direct[:, ok] - want[:, ok]).max() <= 1e-12 * scale
        assert np.all(direct[:, ~ok] == 0)


def test_example_recording_known_answer(golden):
    """The reference's only shipped known answer: matlab_filtered.npy."""
    g = golden("example_dbs")
    data = np.load(get_example_data_paths("example_data"))
    matlab = np.load(get_example_data_paths("matlab_filtered"))
    assert sha(data) == str(g["data_sha256"])
    np.testing.assert_array_equal(matlab, g["matlab_filtered"])
    filt = oracle.build_filter(float(g["period"]), 0.01, 2000, 20, "both")
    np.testing.assert_array_equal(filt, g["filter"])
    out = oracle.apply_filter_fft(data, filt)
    np.testing.assert_array_equal(out, g["filtered"])
    assert np.allclose(out, matlab) and np.abs(out - matlab).max() < 1e-13
    direct = oracle.apply_filter_direct(data, g["taps"])
    assert np.abs(direct - matlab).max() < 1e-13
    hw = oracle.default_half_width(float(g["period"]), float(g["default_period_half_width"]), 0,
                                   data.shape[1])
    assert hw == int(g["default_half_width"])


def test_search_stages_match_reference(golden):
    """Indices, candidate grids and a sample of grid errors of the bundled recording."""
    g = golden("example_dbs")
    data = np.load(get_example_data_paths("example_data"))
    z = oracle.standardise(data, 3.0)
    search = np.arange(data.shape[1] - 1)
    rng = np.random.default_rng(None)
    calls = g["calls"]
    cursor = 0
    for run, (use_n, ignore, bw) in enumerate(oracle.run_plan(search.shape[0])):
        idx = oracle.centre_indices(search, data.shape[1], use_n, ignore, rng)
        np.testing.assert_array_equal(idx, g[f"run{run}_indices"])
        periods = oracle.candidate_periods(tuple(g[f"run{run}_estimate"]), run + 1)
        np.testing.assert_array_equal(periods, g[f"run{run}_periods"])
        block = calls[cursor : cursor + len(periods)]  # the grid stage of this run
        np.testing.assert_array_equal(block[:, 0], periods)
        assert int(block[0, 1]) == min(bw, idx.shape[0] // 4)
        pick = np.arange(0, len(periods), 29)
        got = oracle.objective_many(periods[pick], z, idx, int(block[0, 1]), 1.0)
        np.testing.assert_allclose(got, block[pick, 4], rtol=1e-12)
        same_stage = (calls[:, 1] == block[0, 1]) & (calls[:, 2] == 1.0) & (calls[:, 3] == block[0, 3])
        cursor += int(np.sum(same_stage))


def test_random_index_branch(golden):
    g = golden("synthetic_2x30000")
    n_chans, n, fs, fa, seed = (int(v) for v in g["recording"])
    data = make_recording(n_chans, n, fs, fa, seed=seed)
    assert sha(data) == str(g["data_sha256"])
    assert sha(oracle.standardise(data, 3.0)) == str(g["standard_data_sha256"])
    search = np.arange(n - 1)
    rng = np.random.default_rng(0)
    for run, (use_n, ignore, bw) in enumerate(oracle.run_plan(search.shape[0])):
        idx = oracle.centre_indices(search, n, use_n, ignore, rng)
        np.testing.assert_array_equal(idx, g[f"run{run}_indices"])


@pytest.mark.parametrize("name", ["synthetic_2x30000"])
def test_find_period_end_to_end(golden, name):
    """Whole search through the oracle reproduces the reference's period bit for bit."""
    g = golden(name)
    n_chans, n, fs, fa, seed = (int(v) for v in g["recording"])
    data = make_recording(n_chans, n, fs, fa, seed=seed)
    period = oracle.find_period(data, fs, fa, random_seed=0, n_jobs=8)
    assert period == g["period"]
    for direction in DIRECTIONS:
        hw = int(g["default_half_width"])
        taps = oracle.tap_offsets(period, period / 50, hw, 0, direction)
        np.testing.assert_array_equal(taps, g[f"{direction}_taps"])
        filt = oracle.build_filter(period, period / 50, hw, 0, direction)
        cols = g[f"{direction}_filtered_cols"]
        np.testing.assert_array_equal(oracle.apply_filter_fft(data, filt)[:, cols],
                                      g[f"{direction}_filtered"])


def test_periodogram_matches_reference_compute_psd(golden):
    """oracle.periodogram vs the reference's compute_psd outputs (tests/golden/psd.npz)."""
    g = golden("psd")
    for k in range(int(g["n_cases"])):
        fs, n, fmax = g[f"case{k}_args"]
        freqs, psd = oracle.periodogram(g[f"case{k}_x"], fs, int(n), None if fmax < 0 else fmax)
        want = g[f"case{k}_psd"]
        assert np.array_equal(freqs, g[f"case{k}_freqs"])
        assert psd.dtype == np.float32 and psd.shape == want.shape
        assert np.abs(psd - want).max() <= 1e-5 * np.abs(want).max()

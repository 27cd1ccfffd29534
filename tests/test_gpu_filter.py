"""CUDA period filter vs the reference's recorded outputs, the oracle, and properties.

Tolerance (BASELINE.json north_star): float64 relative error <= 1e-9, float32 mode <= 1e-4,
measured against the largest input magnitude of the recording.  Samples with no tap in range
(SURVEY S2: the reference's FFT path returns rounding noise there) are compared with the
documented intent, 0.
"""

import numpy as np
import pytest

from oracle import parrm_oracle as oracle
from oracle.golden_inputs import checked_filter_edges_inputs
from pyparrm_b200 import PARRM, get_example_data_paths, pinned_empty
from pyparrm_b200.synthetic import make_recording

from pyparrm_b200 import _native

pytestmark = pytest.mark.gpu
RTOL64, RTOL32 = 1e-9, 1e-4
# The planner may regroup the tap sum (comb boxes, filter_plan.h); both evaluation orders are
# checked.  They agree with the oracle's tap-by-tap sum to rounding (<= 1e-13 of the input
# scale), far inside the 1e-9 contract.
STRATEGIES = [_native.PLAN_GATHER, _native.PLAN_AUTO]


def rel_err(got, want, scale):
    return float(np.abs(got - want).max() / scale) if got.size else 0.0


def check_against_reference(got, want_ref, x, taps, rtol=RTOL64, cols=None):
    """``want_ref`` holds the reference's output at columns ``cols`` only, when they are given."""
    ok = oracle.in_range_tap_count(x.shape[1], taps) > 0
    scale = max(np.abs(x).max(), 1e-300)
    assert np.all(got[:, ~ok] == 0)
    if cols is not None:
        got, ok = got[:, cols], ok[cols]
    if ok.any():
        assert rel_err(got[:, ok], want_ref[:, ok], scale) <= rtol


def test_known_answer_matlab(golden, gpu_engine):
    g = golden("example_dbs")
    data = np.load(get_example_data_paths("example_data"))
    out = gpu_engine.filter_host(data, g["taps"])
    assert out.dtype == np.float64 and out.shape == data.shape
    assert np.allclose(out, g["matlab_filtered"])          # the reference example's own check
    assert rel_err(out, g["matlab_filtered"], np.abs(data).max()) <= RTOL64
    assert rel_err(out, g["filtered"], np.abs(data).max()) <= RTOL64
    out_default = gpu_engine.filter_host(data, g["default_taps"])  # 1000 taps
    assert rel_err(out_default, g["default_filtered"], np.abs(data).max()) <= RTOL64


@pytest.mark.parametrize("strategy", STRATEGIES)
def test_synthetic_all_directions(golden, gpu_engine, strategy):
    g = golden("synthetic_2x30000")
    n_chans, n, fs, fa, seed = (int(v) for v in g["recording"])
    data = make_recording(n_chans, n, fs, fa, seed=seed)
    for name in ("both", "past", "future", "hw2000"):
        out = gpu_engine.filter_host(data, g[f"{name}_taps"], strategy=strategy)
        check_against_reference(out, g[f"{name}_filtered"], data, g[f"{name}_taps"],
                                cols=g[f"{name}_filtered_cols"])


@pytest.mark.parametrize("strategy", STRATEGIES)
def test_short_and_ragged_inputs(golden, gpu_engine, strategy):
    g = golden("filter_edges")
    for case, x in enumerate(checked_filter_edges_inputs(g)):
        taps = g[f"case{case}_taps"]
        out = gpu_engine.filter_host(x, taps, strategy=strategy)
        assert out.shape == x.shape
        check_against_reference(out, g[f"case{case}_y"], x, taps)


@pytest.mark.parametrize("strategy", STRATEGIES)
@pytest.mark.parametrize("shape", [(1, 1), (1, 2), (3, 17), (2, 1023), (5, 4096), (1, 4097),
                                   (2, 12289), (7, 20001), (0, 10), (2, 0)])
def test_random_shapes_against_oracle(gpu_engine, shape, strategy):
    rng = np.random.default_rng(shape[0] * 131 + shape[1])
    x = rng.standard_normal(shape) * 3 + 100.0
    per = 15.3846
    for direction, hw, omit in (("both", 2000, 0), ("past", 777, 3), ("future", 50, 0)):
        taps = oracle.tap_offsets(per, per / 50, hw, omit, direction)
        out = gpu_engine.filter_host(x, taps, strategy=strategy)
        want = oracle.apply_filter_direct(x, taps)
        assert out.shape == x.shape
        if x.size:
            assert rel_err(out, want, np.abs(x).max()) <= 1e-13


def test_huge_span_uses_global_gather(gpu_engine):
    """Tap windows too wide for shared memory take the global-memory kernel."""
    rng = np.random.default_rng(1)
    x = rng.standard_normal((2, 90_000))
    taps = oracle.tap_offsets(230.77, 4.6, 40_000, 0, "both")
    out = gpu_engine.filter_host(x, taps)
    assert rel_err(out, oracle.apply_filter_direct(x, taps), np.abs(x).max()) <= 1e-13


def test_pinned_and_pageable_inputs_agree(gpu_engine):
    x = make_recording(6, 300_000, 2000, 130, seed=4)
    taps = oracle.tap_offsets(2000 / 130, 0.3, 2000, 0, "both")
    xp = pinned_empty(x.shape)
    xp[:] = x
    a, b = gpu_engine.filter_host(x, taps), gpu_engine.filter_host(xp, taps)
    assert np.array_equal(a, b)
    xf = np.asfortranarray(x)  # non C-contiguous input
    assert np.array_equal(gpu_engine.filter_host(xf, taps), a)
    assert np.array_equal(gpu_engine.filter_host(x.astype(np.float32), taps),
                          gpu_engine.filter_host(x.astype(np.float32).astype(np.float64), taps))


def test_time_chunked_host_path(gpu_engine, monkeypatch):
    """Rows longer than the chunk budget are split in time with halos (SURVEY 8(e))."""
    from pyparrm_b200 import _engine

    x = make_recording(2, 200_000, 2000, 130, seed=6)
    taps = oracle.tap_offsets(2000 / 130, 0.3, 2000, 0, "both")
    whole = gpu_engine.filter_host(x, taps, strategy=_native.PLAN_GATHER)
    whole_comb = gpu_engine.filter_host(x, taps)
    monkeypatch.setattr(_engine, "_CHUNK_BYTES", 256 << 10)
    chunked = gpu_engine.filter_host(x, taps, strategy=_native.PLAN_GATHER)
    assert np.array_equal(whole, chunked)
    # strips start at other samples when the host chunks in time: equal to rounding only
    chunked_comb = gpu_engine.filter_host(x, taps)
    assert rel_err(chunked_comb, whole_comb, np.abs(x).max()) <= 1e-13
    assert rel_err(whole_comb, whole, np.abs(x).max()) <= 1e-13
    for direction in ("past", "future"):
        t1 = oracle.tap_offsets(2000 / 130, 0.3, 1500, 0, direction)
        assert rel_err(gpu_engine.filter_host(x, t1), oracle.apply_filter_direct(x, t1), 10) <= 1e-13


def test_device_tensor_entry_point(gpu_engine):
    import torch

    x = make_recording(3, 50_000, 2000, 130, seed=8)
    taps = oracle.tap_offsets(2000 / 130, 0.3, 2000, 0, "both")
    d_out = gpu_engine.filter_device(torch.from_numpy(x).cuda(), taps)
    assert rel_err(d_out.cpu().numpy(), oracle.apply_filter_direct(x, taps), 10) <= 1e-13


def test_public_api_accepts_device_tensors(gpu_engine):
    """``PARRM.filter_data(cuda_tensor)`` (additive overload, SURVEY 8(f).2): filtered on the
    device, device tensor back, same values as the NumPy path; other non-NumPy inputs keep the
    reference's TypeError (parrm.py:877-886)."""
    import torch

    data = make_recording(5, 60_000, 2000, 130, seed=2)
    parrm = PARRM(data, 2000, 130, verbose=False)
    parrm._period = np.float64(2000 / 130 * (1 + 3e-6))
    parrm.create_filter(filter_half_width=2000)
    want = parrm.filter_data().copy()
    got = parrm.filter_data(torch.from_numpy(data).cuda())
    assert isinstance(got, torch.Tensor) and got.is_cuda and got.dtype == torch.float64
    assert parrm.filtered_data is got
    assert rel_err(got.cpu().numpy(), want, np.abs(data).max()) <= 1e-13
    got32 = parrm.filter_data(torch.from_numpy(data.astype(np.float32)).cuda())  # widened
    assert got32.dtype == torch.float64
    assert rel_err(got32.cpu().numpy(), want, np.abs(data).max()) <= 1e-6
    strided = torch.from_numpy(np.ascontiguousarray(data.T)).cuda().T  # not row-major
    assert rel_err(parrm.filter_data(strided).cpu().numpy(), want, np.abs(data).max()) <= 1e-13
    with pytest.raises(ValueError, match="must be a 2D array"):
        parrm.filter_data(torch.zeros(7, device="cuda", dtype=torch.float64))
    with pytest.raises(TypeError, match="must be a NumPy array"):
        parrm.filter_data(torch.zeros((2, 7), dtype=torch.float64))  # CPU tensor: reference rule
    with pytest.raises(TypeError, match="must be a NumPy array"):
        parrm.filter_data([[1.0, 2.0]])


def test_float32_mode(gpu_engine):
    x = make_recording(4, 100_000, 2000, 130, seed=9)
    taps = oracle.tap_offsets(2000 / 130, 0.3, 2000, 0, "both")
    out = gpu_engine.filter_host(x, taps, precision="fp32")
    assert out.dtype == np.float64
    assert rel_err(out, oracle.apply_filter_direct(x, taps), np.abs(x).max()) <= RTOL32


def test_full_size_properties(gpu_engine):
    """cfg2 size (64 x 1.2 M, 160 taps): the oracle on a channel subset + exact properties."""
    import torch

    fs, fa, n = 2000, 130, 1_200_000
    x = make_recording(64, n, fs, fa, seed=0)
    per = fs / fa * (1 + 3e-6)
    taps = oracle.tap_offsets(per, per / 50, 2000, 0, "both")
    assert taps.shape[0] == 160
    out = gpu_engine.filter_host(x, taps)
    pick = [0, 31, 63]
    want = oracle.apply_filter_direct(x[pick], taps)
    assert rel_err(out[pick], want, np.abs(x).max()) <= 1e-13
    d_x = torch.from_numpy(x).cuda()
    d_y = gpu_engine.filter_device(d_x, taps)
    # device path == host pipeline (to rounding: the strips start at different samples)
    assert rel_err(d_y.cpu().numpy(), out, np.abs(x).max()) <= 1e-13
    d_g = gpu_engine.filter_device(d_x, taps, strategy=_native.PLAN_GATHER)
    assert rel_err(d_g.cpu().numpy(), out, np.abs(x).max()) <= 1e-13
    # a constant is annihilated wherever a tap is in range; shifts do not change the output
    d_shift = gpu_engine.filter_device(d_x + 1000.0, taps)
    assert float((d_shift - d_y).abs().max()) <= 1e-9
    d_const = gpu_engine.filter_device(torch.full_like(d_x[:2], 7.5), taps)
    assert float(d_const.abs().max()) <= 1e-12
    # linearity
    d_lin = gpu_engine.filter_device(2.5 * d_x[:8] + d_x[8:16], taps)
    assert float((d_lin - (2.5 * d_y[:8] + d_y[8:16])).abs().max()) <= 1e-10
    # the injected artefact (period-locked, 5 harmonics) is removed: what is left is noise-sized
    assert float(d_y[:, 4000:-4000].std()) < 1.15


def test_public_api_filter_matches_golden(golden, gpu_engine):
    g = golden("example_dbs")
    data = np.load(get_example_data_paths("example_data"))
    parrm = PARRM(data, 200, 150, verbose=False)
    parrm._period = np.float64(g["period"])
    parrm.create_filter(filter_half_width=2000, omit_n_samples=20, filter_direction="both",
                        period_half_width=0.01)
    assert np.array_equal(parrm.filter, g["filter"])
    out = parrm.filter_data()
    assert out is parrm.filtered_data
    assert np.allclose(out, g["matlab_filtered"])
    parrm.create_filter()
    assert parrm._filter_half_width == int(g["default_half_width"])
    assert np.array_equal(np.flatnonzero(parrm.filter < 0) - parrm._filter_half_width,
                          g["default_taps"])


def test_time_shards_stitch_to_the_whole(gpu_engine):
    """SURVEY 8(e): fewer channels than GPUs -> time chunks with halos.  The shards of all
    ranks (run one after the other on this GPU) stitch to the unsharded result."""
    from pyparrm_b200 import _sharding

    x = make_recording(1, 123_457, 2000, 130, seed=11)
    for direction in ("both", "past", "future"):
        taps = oracle.tap_offsets(2000 / 130, 0.3, 2000, 0, direction)
        want = oracle.apply_filter_direct(x, taps)
        w_lo, w_hi = min(int(taps[0]), 0), max(int(taps[-1]), 0)
        got = np.full_like(x, np.nan)
        for c0, c1, t0, t1, x0, x1 in _sharding.channel_or_time_shards(1, x.shape[1], 4, w_lo, w_hi):
            got[c0:c1, t0:t1] = gpu_engine.filter_host_window(x[c0:c1, x0:x1], taps, x0, t0, t1,
                                                              x.shape[1])
        assert rel_err(got, want, np.abs(x).max()) <= 1e-13


@pytest.mark.parametrize("name, fs, fa, n_chans, n, hw, direction", [
    ("cfg3 ECoG 1 kHz / 145 Hz, default half-width", 1000, 145, 6, 400_000, 2469, "both"),
    ("cfg4 Neuropixels-like 30 kHz / 130 Hz, causal", 30000, 130, 6, 600_000, 2311, "past"),
    ("cfg4, the other one-sided direction", 30000, 130, 3, 300_000, 2311, "future"),
])
def test_baseline_config_shapes(gpu_engine, name, fs, fa, n_chans, n, hw, direction):
    """The tap structures of BASELINE configs 3 and 4 (stride 200 with windows 25/12; stride 1
    runs of 9 consecutive taps) at reduced channel counts, against the oracle and the plain
    gather kernel."""
    x = make_recording(n_chans, n, fs, fa, seed=17)
    per = fs / fa * (1 + 3e-6)
    taps = oracle.tap_offsets(per, per / 50, hw, 0, direction)
    _, desc = _native.plan_filter(taps)
    assert desc["kind"] == 1, name
    out = gpu_engine.filter_host(x, taps)
    ref = gpu_engine.filter_host(x, taps, strategy=_native.PLAN_GATHER)
    assert rel_err(out, ref, np.abs(x).max()) <= 1e-13
    want = oracle.apply_filter_direct(x[:2], taps)
    assert rel_err(out[:2], want, np.abs(x).max()) <= 1e-13
    assert rel_err(ref[:2], want, np.abs(x).max()) <= 1e-13


# ---------------------------------------------------------------------------------------------
# Run-time specialised kernel (filter_comb_e.cuh through NVRTC), forced at small sizes
SPECIALISED_CASES = {
    "cfg2": (2000 / 130 * (1 + 3e-6), None, 2000, 0, "both"),
    "cfg3": (1000 / 145 * (1 + 3e-6), None, 2469, 0, "both"),
    "cfg4 past": (30000 / 130 * (1 + 3e-6), None, 2311, 0, "past"),
    "cfg4 future": (30000 / 130 * (1 + 3e-6), None, 2311, 0, "future"),
    "cfg1": (1.3311148014466094, 0.01, 2000, 20, "both"),
    "cfg2 past, omit": (2000 / 130 * (1 + 3e-6), None, 1500, 300, "past"),
    # tap structures away from the BASELINE configs: the bundled example with create_filter()'s
    # defaults (period 1.33 samples), a non-integer period with long windows, runs of
    # consecutive taps (wide period_half_width), a short one-sided filter
    "example default": (1.3311148014466094, None, 2408, 0, "both"),
    "ecog-like": (8.6613, None, 5000, 0, "both"),
    "wide runs": (2000 / 130, 1.0, 2000, 0, "both"),
    "wide runs past": (30000 / 130, 20.0, 5000, 0, "past"),
    "short future": (7.3, 0.5, 300, 5, "future"),
}


def _case_taps(name):
    period, phw, hw, omit, direction = SPECIALISED_CASES[name]
    return oracle.tap_offsets(period, period / 50 if phw is None else phw, hw, omit, direction)


@pytest.mark.parametrize("name", list(SPECIALISED_CASES))
def test_specialised_kernel_against_oracle(gpu_engine, name):
    """Interior blocks, recording edges, recordings shorter than the tap window, one strip and
    many strips -- against the oracle's tap-by-tap sum, and fp32 storage within 1e-4."""
    import torch

    taps = _case_taps(name)
    rng = np.random.default_rng(len(name))
    for shape in [(3, 50_000), (1, 7001), (2, 1999), (5, 20_011), (160, 30_000)]:
        x = rng.standard_normal(shape) * 3 + 10
        want = oracle.apply_filter_direct(x, taps)
        d_x = torch.from_numpy(x).cuda()
        got = gpu_engine.filter_device(d_x, taps, kernel=_native.KERNEL_SPECIALISED)
        assert gpu_engine.last_filter_kernel == "parrm_filter_comb_e"
        # rounding of both sums grows with the number of taps (860 in the widest case)
        tol = max(1e-13, 2.5e-16 * len(taps))
        assert rel_err(got.cpu().numpy(), want, np.abs(x).max()) <= tol, (name, shape)
    got32 = gpu_engine.filter_device(d_x.float(), taps, kernel=_native.KERNEL_SPECIALISED)
    assert rel_err(got32.double().cpu().numpy(), want, np.abs(x).max()) <= RTOL32


def test_specialised_kernel_alignment_and_windows(gpu_engine):
    """Rows that start on odd elements (the TMA source must be 16-byte aligned: the chunk grid
    shifts per row) and output ranges inside a longer recording (time shards)."""
    import torch

    taps = _case_taps("cfg2")
    rng = np.random.default_rng(5)
    x = rng.standard_normal((4, 30_001))
    buf = torch.zeros(4 * 30_003 + 1, dtype=torch.float64, device="cuda")
    d_x = buf[1:].as_strided((4, 30_001), (30_003, 1))
    d_x.copy_(torch.from_numpy(x))
    got = gpu_engine.filter_device(d_x, taps, kernel=_native.KERNEL_SPECIALISED).cpu().numpy()
    assert rel_err(got, oracle.apply_filter_direct(x, taps), np.abs(x).max()) <= 1e-13
    # time shard through the C ABI's x_t0 / t0 / n_out arguments, specialised kernel forced
    import os

    x = make_recording(1, 200_003, 2000, 130, seed=3)
    want = oracle.apply_filter_direct(x, taps)
    os.environ["PYPARRM_B200_FILTER_KERNEL"] = str(_native.KERNEL_SPECIALISED)
    try:
        for t0, t1 in ((0, 70_001), (70_001, 150_000), (150_000, 200_003)):
            x0, x1 = max(0, t0 - 2000), min(x.shape[1], t1 + 2000)
            got = gpu_engine.filter_host_window(x[:, x0:x1], taps, x0, t0, t1, x.shape[1])
            assert gpu_engine.last_filter_kernel == "parrm_filter_comb_e"
            assert rel_err(got, want[:, t0:t1], np.abs(x).max()) <= 1e-13
    finally:
        del os.environ["PYPARRM_B200_FILTER_KERNEL"]


@pytest.mark.parametrize("name", ["cfg2", "cfg4 past"])
def test_non_finite_samples_zero_their_window_only(gpu_engine, name):
    """parrm.py:869 replaces non-finite outputs by 0.  Here a NaN / Inf sample zeroes exactly
    the outputs whose tap window (or own sample) contains it -- in both kernels -- and every
    other output is unaffected; a 1e12 outlier only costs rounding.  (The reference's FFT
    convolution spreads one NaN over the whole channel and so zeroes the channel: the
    per-output rule is what its isfinite test expresses.)"""
    import torch

    taps = _case_taps(name)
    rng = np.random.default_rng(9)
    x = rng.standard_normal((3, 60_000))
    x[0, 12_345] = np.nan
    x[1, 30_000] = np.inf
    x[1, 30_007] = -np.inf
    x[2, 5] = 1e12
    with np.errstate(invalid="ignore"):
        want = oracle.apply_filter_direct(x, taps)
    want[~np.isfinite(want)] = 0.0
    d_x = torch.from_numpy(x).cuda()
    outs = {}
    for kern in (_native.KERNEL_SPECIALISED, _native.KERNEL_GATHER):
        got = gpu_engine.filter_device(d_x, taps, kernel=kern).cpu().numpy()
        assert np.isfinite(got).all()
        assert np.array_equal(got[:2] == 0, want[:2] == 0), gpu_engine.last_filter_kernel
        assert np.abs(got[:2] - want[:2]).max() <= 1e-12
        assert np.abs(got[2] - want[2]).max() <= 1e-3       # rounding of a 1e12 outlier
        assert np.abs(got[2, 10_000:] - want[2, 10_000:]).max() <= 1e-12   # gone past its window
        outs[kern] = got
    assert np.array_equal(outs[_native.KERNEL_SPECIALISED][:2] == 0,
                          outs[_native.KERNEL_GATHER][:2] == 0)


def test_storage_dtypes_cross_pcie_as_they_are(gpu_engine):
    """float32 / int16 / int32 recordings are uploaded in their own width and widened on the
    device; the result equals filtering the widened recording (the reference widens on the
    host, parrm.py:861-866).  ``out_dtype=float32`` and the fp32 mode stay within 1e-4."""
    from pyparrm_b200 import pin_array

    taps = _case_taps("cfg2")
    rng = np.random.default_rng(2)
    base = rng.standard_normal((5, 40_000)) * 300
    for dtype in (np.float32, np.int16, np.int32, np.int64, np.float64):
        x = base.astype(dtype)
        want = oracle.apply_filter_direct(x.astype(np.float64), taps)
        out = gpu_engine.filter_host(x, taps)
        assert out.dtype == np.float64
        assert rel_err(out, want, np.abs(base).max()) <= 1e-13, dtype
        out32 = gpu_engine.filter_host(x, taps, out_dtype=np.float32)
        assert out32.dtype == np.float32
        assert rel_err(out32.astype(np.float64), want, np.abs(base).max()) <= RTOL32
        fast = gpu_engine.filter_host(x, taps, precision="fp32", out_dtype=np.float32)
        assert rel_err(fast.astype(np.float64), want, np.abs(base).max()) <= RTOL32
    # registering the caller's array in place: same numbers, direct copies
    x = base.copy()
    with pin_array(x) as pinned:
        from pyparrm_b200._engine import is_pinned

        assert is_pinned(pinned)
        out = gpu_engine.filter_host(pinned, taps)
    assert rel_err(out, oracle.apply_filter_direct(base, taps), np.abs(base).max()) <= 1e-13
    parrm = PARRM(base.astype(np.int16), 2000, 130, verbose=False)
    parrm._period = np.float64(2000 / 130 * (1 + 3e-6))
    parrm.create_filter(filter_half_width=2000)
    got = parrm.filter_data(out_dtype=np.float32)
    want = oracle.apply_filter_direct(base.astype(np.int16).astype(np.float64), taps)
    assert got.dtype == np.float32 and rel_err(got.astype(np.float64), want, 1e3) <= RTOL32


def test_strip_partition_and_timeline(gpu_engine):
    """Strips of equal cost (the default) and strips of equal length (``variant`` 4) cover every
    output exactly once on a shape whose channels are shorter than a strip.  The two partitions
    start their running sums at different samples, so they agree to rounding (the same 1e-13 of
    the input scale both keep against the oracle), not bit for bit; the per-CTA timeline
    (``variant`` 2 + ``timeline``) keeps the partition, so it is bit-identical, and records one
    row per CTA."""
    import torch

    taps = _case_taps("cfg2")
    rng = np.random.default_rng(11)
    x = rng.standard_normal((37, 64_123))
    d_x = torch.from_numpy(x).cuda()
    base = gpu_engine.filter_device(d_x, taps, kernel=_native.KERNEL_SPECIALISED)
    assert rel_err(base.cpu().numpy(), oracle.apply_filter_direct(x, taps), np.abs(x).max()) <= 1e-13
    equal_length = gpu_engine.filter_device(d_x, taps, kernel=_native.KERNEL_SPECIALISED,
                                            tuning={"variant": 4})
    want = oracle.apply_filter_direct(x, taps)
    assert rel_err(equal_length.cpu().numpy(), want, np.abs(x).max()) <= 1e-13
    assert rel_err(equal_length.cpu().numpy(), base.cpu().numpy(), np.abs(x).max()) <= 1e-13
    timeline = torch.zeros(4 * 1024, dtype=torch.int64, device="cuda")
    timed = gpu_engine.filter_device(d_x, taps, kernel=_native.KERNEL_SPECIALISED,
                                     tuning={"variant": 2, "timeline": timeline.data_ptr()})
    assert torch.equal(base, timed)
    rows = timeline.cpu().numpy().reshape(-1, 4)
    rows = rows[rows[:, 2] > 0]
    assert 1 <= len(rows) <= 2 * 148
    assert (rows[:, 2] >= rows[:, 1]).all() and (rows[:, 0] < 148).all()
    # pieces per CTA: a strip can be empty on a job this small, and some CTA must have worked
    assert (rows[:, 3] >= 0).all() and rows[:, 3].sum() >= 37

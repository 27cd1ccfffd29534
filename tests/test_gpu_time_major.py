"""Time-major recordings on the B200: ``[channels, times]`` views of ``[times, channels]`` arrays
(``mm.T``, ``mm[:, a:b].T``) are filtered, searched and streamed without a host transpose, with
the same results as their C-order twins."""

import tracemalloc

import numpy as np
import pytest

from oracle import parrm_oracle as oracle
from pyparrm_b200 import PARRM, _engine, _native, get_example_data_paths
from pyparrm_b200._engine import pin_array, pinned_empty
from pyparrm_b200._stream import FilterStream
from pyparrm_b200.synthetic import make_recording
from tests.test_gpu_fp32 import CombShape, comb_bound, gather_bound, rounded
from tests.test_gpu_stream_recalibrate import SimpleFilter

pytestmark = pytest.mark.gpu
GATHER = _native.PLAN_GATHER
CODES = {np.dtype(np.float64): _native.F64, np.dtype(np.float32): _native.F32,
         np.dtype(np.int16): _native.I16, np.dtype(np.int32): _native.I32}
STORAGE = [np.float64, np.float32, np.int16, np.int32]


# ---------------------------------------------------------------------------------------------
# 1. parrm_transpose against NumPy
@pytest.mark.parametrize("src_dtype", STORAGE)
def test_transpose_every_pair_shape_pitch_and_offset(gpu_engine, src_dtype):
    import torch

    rng = np.random.default_rng(0)
    src_dtype = np.dtype(src_dtype)
    for dst_dtype in dict.fromkeys([src_dtype, np.dtype(np.float64), np.dtype(np.float32)]):
        for rows, cols in ((1, 1), (1, 300), (300, 1), (64, 64), (67, 129), (130, 65), (3, 1000),
                           (1000, 3), (2049, 385)):
            for src_ld, off in ((cols, 0), (cols + 1, 1), (cols + 7, 2), (cols + 64, 3)):
                if src_dtype.kind == "f":
                    src = rng.standard_normal((rows, src_ld)) * 1e3
                else:
                    src = rng.integers(-30_000, 30_000, (rows, src_ld))
                flat = np.zeros(rows * src_ld + off, dtype=src_dtype)
                flat[off:] = src.astype(src_dtype).ravel()
                d_src = torch.from_numpy(flat).cuda()
                dst_ld = rows + (5 if off else 0)
                d_dst = torch.full((cols, dst_ld), -7, dtype=torch.from_numpy(
                    np.zeros(1, dst_dtype)).dtype, device="cuda")
                _native.check(_native.lib.parrm_transpose(
                    d_src.data_ptr() + off * src_dtype.itemsize, CODES[src_dtype], rows, cols,
                    src_ld, d_dst.data_ptr(), CODES[dst_dtype], dst_ld, None), "parrm_transpose")
                got = d_dst.cpu().numpy()
                want = flat[off:].reshape(rows, src_ld)[:, :cols].T.astype(dst_dtype)
                assert np.array_equal(got[:, :rows], want), (src_dtype, dst_dtype, rows, cols,
                                                             src_ld, off)
                assert np.all(got[:, rows:] == -7)  # nothing written past `rows` in a row


# ---------------------------------------------------------------------------------------------
# 2. filter_data on time-major recordings
TAPS = {"both": oracle.tap_offsets(2000 / 130 * (1 + 3e-6), 2000 / 130 / 50, 60, 0, "both"),
        "past": oracle.tap_offsets(2000 / 130 * (1 + 3e-6), 2000 / 130 / 50, 60, 0, "past")}
N_SAMPLES = 6_000


def recording(dtype, n_chans, ld, first, seed=0, non_finite=False, span=120):
    """(time-major view, C-order twin, [T, ld] base): channels [first, first + n_chans) of the
    base; with ``non_finite`` a NaN inside a window's halo and +-Inf at window boundaries."""
    x = make_recording(ld, N_SAMPLES, 2000, 130, seed=seed) * 300
    dtype = np.dtype(dtype)
    base = np.ascontiguousarray(x.T).astype(dtype)
    if non_finite and dtype.kind == "f":
        step = 16 * span
        base[step - 3, first] = np.nan                          # halo of the second window
        base[2 * step, first + n_chans - 1] = np.inf            # first output of the third
        base[step - 1, first + n_chans // 2] = -np.inf          # last output of the first
    view = base[:, first:first + n_chans].T
    assert _engine.time_major_ld(view) == ld
    return view, np.ascontiguousarray(view), base


# (C, ld, first channel); the last two are 15x and 385x narrower than their rows: the first is
# read as rows, the second (one electrode, or the sync channel) keeps the host copy
LAYOUTS = [(1, 5, 4), (3, 7, 2), (64, 64, 0), (385, 386, 1), (25, 385, 360), (1, 385, 384)]


def run_filter(engine, view, taps, precision, out_dtype, out_mode, pinned, strategy=None):
    n_chans, n = view.shape
    want_dtype = np.dtype(np.float64 if out_dtype is None else out_dtype)
    out = None
    if out_mode == "c":
        out = (pinned_empty((n_chans, n), want_dtype) if pinned
               else np.empty((n_chans, n), want_dtype))
    elif out_mode == "tm":
        base = (pinned_empty((n, n_chans + 2), want_dtype) if pinned
                else np.empty((n, n_chans + 2), want_dtype))
        out = base[:, 1:n_chans + 1].T
    kw = {} if out is None else {"out": out}
    got = engine.filter_host(view, taps, precision, strategy=strategy, out_dtype=out_dtype, **kw)
    if out is not None:
        assert got is out
    assert got.dtype == want_dtype and got.shape == view.shape
    return np.asarray(got)


@pytest.mark.parametrize("precision", ["fp64", "fp32"])
@pytest.mark.parametrize("out_dtype", [None, np.float32])
@pytest.mark.parametrize("dtype", STORAGE)
def test_filter_time_major_is_bit_equal_to_the_c_order_twin(gpu_engine, monkeypatch, dtype,
                                                           out_dtype, precision):
    """Gather plan: every output of a time window equals the whole-row result bit for bit."""
    monkeypatch.setenv("PYPARRM_B200_PLAN", str(GATHER))
    monkeypatch.setattr(_engine, "_CHUNK_BYTES", 1)  # windows of 16 * span: many per recording
    for direction, taps in TAPS.items():
        span = max(int(taps[-1]), 0) - min(int(taps[0]), 0)
        for n_chans, ld, first in LAYOUTS:
            view, twin, base = recording(dtype, n_chans, ld, first, non_finite=True, span=span)
            assert N_SAMPLES > 3 * _engine.window_step(span, ld * 8, n_chans * 8)
            want = gpu_engine.filter_host(twin, taps, precision, out_dtype=out_dtype)
            for pinned in (False, True):
                handle = pin_array(base) if pinned else None
                try:
                    for out_mode in ("default", "c", "tm"):
                        got = run_filter(gpu_engine, view, taps, precision, out_dtype, out_mode,
                                         pinned)
                        assert np.array_equal(got, want, equal_nan=True), (
                            direction, n_chans, pinned, out_mode)
                        # C-order input into an `out`: the same time windows
                        if out_mode != "default":
                            got = run_filter(gpu_engine, twin, taps, precision, out_dtype,
                                             out_mode, pinned)
                            assert np.array_equal(got, want, equal_nan=True)
                finally:
                    if handle is not None:
                        handle.release()


@pytest.mark.parametrize("precision", ["fp64", "fp32"])
@pytest.mark.parametrize("dtype", STORAGE)
def test_filter_time_major_default_plan_against_the_oracle(gpu_engine, monkeypatch, dtype,
                                                           precision):
    """Default (comb) plan, specialised kernel when it applies: held to the oracle."""
    monkeypatch.setattr(_engine, "_CHUNK_BYTES", 1)
    monkeypatch.setenv("PYPARRM_B200_FILTER_KERNEL", "-1")
    for taps in TAPS.values():
        for n_chans, ld, first in LAYOUTS:
            view, twin, base = recording(dtype, n_chans, ld, first, seed=1)
            x64 = twin.astype(np.float64)
            if precision == "fp64":
                want = oracle.apply_filter_direct(x64, taps)
                bound = np.full(want.shape, 1e-13 * np.abs(x64).max())
            else:  # the oracle on the recording as float32 sees it, to the fp32 error models
                xr = rounded(x64)
                want = oracle.apply_filter_direct(xr, taps)
                bound = gather_bound(xr, taps)
                if _native.plan_filter(taps, _native.F32)[1]["kind"] == 1:
                    bound = np.maximum(bound, comb_bound(xr, taps, CombShape(taps),
                                                         np.abs(xr).max()))
            for out_dtype in (None, np.float32):
                # a float32 result of the fp64 mode is rounded once more
                tol = bound + (np.abs(want) * 2.0 ** -24 * 1.01
                               if out_dtype is not None and precision == "fp64" else 0.0)
                for pinned in (False, True):
                    handle = pin_array(base) if pinned else None
                    try:
                        for out_mode in ("default", "c", "tm"):
                            got = run_filter(gpu_engine, view, taps, precision, out_dtype,
                                             out_mode, pinned).astype(np.float64)
                            assert np.all(np.abs(got - want) <= tol), (
                                n_chans, out_dtype, out_mode, pinned)
                    finally:
                        if handle is not None:
                            handle.release()


def test_memmap_round_trip_makes_no_host_copy(gpu_engine, monkeypatch, tmp_path):
    """int16 [T, 385] file in, channels 0..383 filtered into a float32 [T, 384] file."""
    monkeypatch.setenv("PYPARRM_B200_PLAN", str(GATHER))
    n, fs = 120_000, 30000
    x = (make_recording(385, n, fs, 130, seed=5) * 300).astype(np.int16)
    src = tmp_path / "rec.npy"
    np.save(src, np.ascontiguousarray(x.T))
    del x
    mm = np.load(src, mmap_mode="r")
    parrm = PARRM(mm[:, :384].T, fs, 130, verbose=False)
    parrm._period = np.float64(fs / 130 * (1 + 3e-6))
    parrm.create_filter(filter_half_width=600, filter_direction="past")
    dst = tmp_path / "out.npy"
    res = np.lib.format.open_memmap(dst, mode="w+", dtype=np.float32, shape=(n, 384))
    parrm.filter_data()  # warm: plan, ring and staging exist before the measured call
    tracemalloc.start()
    got = parrm.filter_data(out=res.T)
    peak = tracemalloc.get_traced_memory()[1]
    tracemalloc.stop()
    assert got is parrm.filtered_data and np.shares_memory(got, res)
    assert peak < mm[:, :384].nbytes // 4, peak
    res.flush()
    del res, got
    back = np.load(dst)
    want = parrm.filter_data(np.ascontiguousarray(mm[:, :384].T), out_dtype=np.float32)
    assert np.array_equal(back.T, want)


# ---------------------------------------------------------------------------------------------
# 3. find_period on time-major recordings
def fit_errors(parrm):
    seen = []
    orig_first = PARRM._optimise_period_estimate_first_run
    orig_second = PARRM._optimise_period_estimate_second_run

    def first(self, periods, tile, bandwidth, lambda_):
        p, e = orig_first(self, periods, tile, bandwidth, lambda_)
        seen.append(("grid", p.copy(), e.copy()))
        return p, e

    def second(self, periods, errors, tile, bandwidth, lambda_):
        out = orig_second(self, periods, errors, tile, bandwidth, lambda_)
        seen.append(("nm", periods.copy(), errors.copy()))
        return out

    with pytest.MonkeyPatch.context() as mp:
        mp.setattr(PARRM, "_optimise_period_estimate_first_run", first)
        mp.setattr(PARRM, "_optimise_period_estimate_second_run", second)
        parrm.find_period(random_seed=3)
    return parrm.period, seen


def search_cases(dtype):
    """The bundled example (one channel: a column of a [T, 2] array, as ``np.asfortranarray``
    of one channel is C-contiguous too), a Fortran-ordered synthetic and a channel subset."""
    example = np.load(get_example_data_paths("example_data")).astype(dtype)
    base = np.zeros((example.shape[1], 2), dtype=dtype)
    base[:, 0] = example[0]
    yield "example", base[:, :1].T, 200, 150
    synth = make_recording(9, 40_001, 2000, 130, seed=7).astype(dtype)
    yield "fortran", np.asfortranarray(synth), 2000, 130
    yield "subset", np.ascontiguousarray(synth.T)[:, 2:7].T, 2000, 130


@pytest.mark.parametrize("precision", ["fp64", "fp32"])
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_find_period_time_major_is_bit_equal(gpu_engine, monkeypatch, dtype, precision):
    uploads = []
    orig = _engine.DeviceEngine._upload_time_major

    def spy(self, data):
        uploads.append(data.shape)
        return orig(self, data)

    monkeypatch.setattr(_engine.DeviceEngine, "_upload_time_major", spy)
    for name, data, fs, fa in search_cases(dtype):
        assert _engine.time_major_ld(data) is not None, name
        want = fit_errors(PARRM(np.ascontiguousarray(data), fs, fa, verbose=False,
                                precision=precision))
        for share, device in ((0.5, True), (0.0, False)):   # both sides of the memory rule
            monkeypatch.setattr(_engine, "_SEARCH_DEVICE_SHARE", share)
            uploads.clear()
            got = fit_errors(PARRM(data, fs, fa, verbose=False, precision=precision))
            assert bool(uploads) == device, (name, share)
            assert got[0] == want[0], (name, share)
            assert len(got[1]) == len(want[1])
            for (k1, p1, e1), (k2, p2, e2) in zip(got[1], want[1]):
                assert k1 == k2 and np.array_equal(p1, p2) and np.array_equal(e1, e2)


def test_find_period_time_major_chunks(gpu_engine, monkeypatch):
    """Many upload chunks (rows of the base) give the same tiles as one."""
    monkeypatch.setattr(_engine, "_SEARCH_CHUNK_BYTES", 5 * 7 * 8 * 997)
    synth = make_recording(7, 30_003, 2000, 130, seed=2)
    view = np.ascontiguousarray(synth.T)[:, 1:6].T
    want = fit_errors(PARRM(np.ascontiguousarray(view), 2000, 130, verbose=False))
    got = fit_errors(PARRM(view, 2000, 130, verbose=False))
    assert got[0] == want[0]
    for (_, p1, e1), (_, p2, e2) in zip(got[1], want[1]):
        assert np.array_equal(p1, p2) and np.array_equal(e1, e2)


# ---------------------------------------------------------------------------------------------
# 4. streams fed time-major blocks
@pytest.mark.parametrize("graphs", [False, True])
@pytest.mark.parametrize("dtype", [np.int16, np.float32, np.float64])
def test_stream_time_major_blocks_across_a_switch(gpu_engine, dtype, graphs):
    period = 30000 / 130 * (1 + 3e-6)
    taps_a = oracle.tap_offsets(period, period / 50, 2311, 0, "future")
    taps_b = oracle.tap_offsets(30000 / 131, 30000 / 131 / 50, 1500, 0, "both")
    x = make_recording(385, 40_000, 30000, 130, seed=4) * 50
    base = np.ascontiguousarray(x.T).astype(dtype)       # frames as acquisition delivers them
    sizes = [300] * 40 + [1, 13, 5000, 3001, 300, 300] + [300] * 30
    sizes.append(base.shape[0] - sum(sizes))
    outs = {}
    for layout in ("c", "tm"):
        stream = FilterStream(gpu_engine, taps_a, max_chunk=4096, graphs=graphs, history=6_000)
        got, t = [], 0
        for i, n in enumerate(sizes):
            if i == 45:
                stream.set_filter(SimpleFilter(taps_b))
            frame = base[t:t + n, :384]
            block = frame.T if layout == "tm" else np.ascontiguousarray(frame.T)
            if layout == "tm" and n > 1:
                assert _engine.time_major_ld(block) == 385
            got.append(stream.push(block))
            t += n
        got.append(stream.close())
        outs[layout] = np.concatenate(got, axis=1)
    assert np.array_equal(outs["tm"], outs["c"])


def test_views_much_narrower_than_their_rows_keep_the_host_copy(gpu_engine, monkeypatch):
    """filter_data, find_period and stream pushes transpose on the device exactly when
    ``time_major_input_ld`` says so; the sync channel of a 385-channel file is copied on the
    host, as before, instead of uploading all 385 channels."""
    calls = []
    real = _native.lib.parrm_transpose

    def counting(*args):
        calls.append(args[2:5])
        return real(*args)

    monkeypatch.setattr(_native.lib, "parrm_transpose", counting)
    monkeypatch.setenv("PYPARRM_B200_PLAN", str(GATHER))
    taps = TAPS["past"]
    base = np.ascontiguousarray((make_recording(385, 20_000, 2000, 130, seed=9) * 300).T)
    for lo, hi, rows in ((384, 385, False), (380, 385, False), (375, 385, True), (0, 384, True)):
        view = base[:, lo:hi].T
        assert (_engine.time_major_input_ld(view) is not None) == rows
        for kind in ("filter", "search", "stream"):
            calls.clear()
            if kind == "filter":
                got = gpu_engine.filter_host(view, taps)
                assert np.array_equal(got, gpu_engine.filter_host(np.ascontiguousarray(view),
                                                                  taps))
            elif kind == "search":
                parrm = PARRM(view, 2000, 130, verbose=False)
                twin = PARRM(np.ascontiguousarray(view), 2000, 130, verbose=False)
                parrm.find_period(random_seed=1)
                n_calls = len(calls)
                twin.find_period(random_seed=1)
                calls[n_calls:] = []
                assert parrm.period == twin.period
            else:
                stream = FilterStream(gpu_engine, taps, max_chunk=4096)
                got = np.concatenate([stream.push(view[:, t:t + 3000])
                                      for t in range(0, 20_000, 3000)] + [stream.close()], axis=1)
                assert np.array_equal(got, gpu_engine.filter_host(np.ascontiguousarray(view), taps,
                                                                  strategy=GATHER))
            assert bool(calls) == rows, (lo, hi, kind)
            assert all(ld == 385 for _, _, ld in calls)

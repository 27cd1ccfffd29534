"""Re-calibrating an open stream on the B200: switched streams are bit-equal to the gather filter
over each tap set's range of outputs, ``recent()`` hands back the ring's samples, and a
``PARRM`` built on a CUDA tensor finds the same period, bit for bit, as its NumPy twin without
crossing PCIe."""

import threading

import numpy as np
import pytest

from oracle import parrm_oracle as oracle
from pyparrm_b200 import PARRM, _engine, _native
from pyparrm_b200._stream import FilterStream
from pyparrm_b200.synthetic import make_recording
from tests.test_stream_recalibrate_logic import (
    CHANGE, DRIFT, F_NEW, FS, frequency_change_recording)

pytestmark = pytest.mark.gpu
GATHER = _native.PLAN_GATHER
COPIES = ("parrm_copy_h2d_async", "parrm_copy_d2h_async", "parrm_host_copy")


def to_np(y):
    return y.cpu().numpy() if hasattr(y, "is_cuda") else y


def run_switched(engine, taps_list, x, sizes, at, ref=None, **kw):
    """Push ``x`` in ``sizes`` blocks; before push ``at[k]`` switch to ``taps_list[k + 1]``.
    Returns the outputs and the per-segment gather reference on ``ref`` (the NumPy twin of a
    CUDA ``x``)."""
    stream = FilterStream(engine, taps_list[0], **kw)
    outs, segments, t = [], [(0, taps_list[0])], 0
    for i, n in enumerate(sizes + [None]):
        if i in at:
            taps = taps_list[at.index(i) + 1]
            stream.set_filter(SimpleFilter(taps))
            segments.append((stream.n_emitted, taps))
        y = stream.close() if n is None else stream.push(x[:, t:t + n])
        t += 0 if n is None else n
        outs.append(to_np(y))
        assert stream.n_emitted == sum(o.shape[1] for o in outs)
    got = np.concatenate(outs, axis=1)
    host = x if ref is None else ref
    bounds = [s for s, _ in segments[1:]] + [x.shape[1]]
    want = np.concatenate([
        engine.filter_host(host, taps, precision=kw.get("precision", "fp64"), strategy=GATHER,
                           out_dtype=kw.get("out_dtype"))[:, s:s1]
        for (s, taps), s1 in zip(segments, bounds)], axis=1)
    return got, want


class SimpleFilter:
    """What ``set_filter`` reads of a PARRM object: ``_filter`` and ``_tap_offsets()``."""

    def __init__(self, taps):
        self._taps = np.asarray(taps, dtype=np.int32)
        self._filter = np.zeros(1)

    def _tap_offsets(self):
        return self._taps


def taps_of(direction, hw, period=30000 / 130 * (1 + 3e-6)):
    return oracle.tap_offsets(period, period / 50, hw, 0, direction)


def sizes_of(seed, total):
    rng = np.random.default_rng(seed)
    sizes = []
    while sum(sizes) < total:
        sizes.append(int(rng.choice([1, 13, 300, 301, 997, 3000, 5000])))
    sizes[-1] -= sum(sizes) - total
    return [s for s in sizes if s > 0]


@pytest.mark.parametrize("kind", ["float64", "fp32", "int16", "cuda", "cuda_int16"])
def test_switch_is_bit_equal_to_the_per_segment_gather_filter(gpu_engine, kind):
    import torch

    x = make_recording(6, 60_000, 30000, 130, seed=4) * 50
    if kind in ("int16", "cuda_int16"):
        x = x.astype(np.int16)
    kw = {"precision": "fp32"} if kind == "fp32" else {}
    taps_list = [taps_of("future", 2311), taps_of("both", 1500, 30000 / 131),
                 taps_of("past", 2000, 30000 / 129), taps_of("future", 900)]
    for seed in range(2):
        sizes = sizes_of(seed, x.shape[1])
        at = [0] + sorted(np.random.default_rng(seed).choice(
            np.arange(1, len(sizes)), 2, replace=False).tolist())
        data = torch.from_numpy(x).cuda() if kind.startswith("cuda") else x
        got, want = run_switched(gpu_engine, taps_list, data, sizes, at, ref=x, history=6_000,
                                 max_chunk=4096, **kw)
        assert np.array_equal(got, want), (kind, seed)


def test_switch_with_a_span_that_needs_the_global_kernel(gpu_engine):
    rng = np.random.default_rng(1)
    x = rng.standard_normal((2, 200_000))
    wide = oracle.tap_offsets(230.77, 4.6, 40_000, 0, "both")
    narrow = oracle.tap_offsets(229.9, 4.6, 2_000, 0, "past")
    assert (max(int(wide[-1]), 0) - int(wide[0])) * 8 > 200 * 1024
    sizes = [1, 30_011, 65_536, 7, 41_000, 63_445]
    for taps_list in ([narrow, wide], [wide, narrow]):
        got, want = run_switched(gpu_engine, taps_list, x, sizes, [3], history=82_000)
        assert np.array_equal(got, want)


def test_graph_replay_before_and_after_a_switch(gpu_engine):
    x = (make_recording(16, 60_000, 30000, 130, seed=3) * 50).astype(np.int16)
    taps_list = [taps_of("future", 2311), taps_of("both", 2000, 30000 / 131)]
    sizes = [300] * 200
    got, want = run_switched(gpu_engine, taps_list, x, sizes, [100], out_dtype=np.float32,
                             graphs=True, history=5_000)
    assert np.array_equal(got, want)
    eager, _ = run_switched(gpu_engine, taps_list, x, sizes, [100], out_dtype=np.float32,
                            history=5_000)
    assert np.array_equal(got, eager)


def test_recent_returns_the_pushed_samples_widened(gpu_engine):
    import torch

    rng = np.random.default_rng(2)
    x = rng.integers(-30_000, 30_000, (5, 50_000)).astype(np.int16)
    taps = taps_of("future", 300)
    for precision, dtype in (("fp64", torch.float64), ("fp32", torch.float32)):
        for data in (x, torch.from_numpy(x).cuda()):
            stream = FilterStream(gpu_engine, taps, precision=precision, max_chunk=1_000,
                                  history=7_000)
            t = 0
            for n in (3_000, 2_500, 7_001, 13, 9_999):  # pushes split by max_chunk; ring wraps
                stream.push(data[:, t:t + n])
                t += n
                for k in (1, 777, min(t, 7_000)):
                    got = stream.recent(k)
                    assert got.is_cuda and got.dtype == dtype and got.shape == (5, k)
                    assert np.array_equal(got.cpu().numpy(), x[:, t - k:t].astype(
                        np.float32 if precision == "fp32" else np.float64))
            stream.close()


def test_pushes_do_not_wait_for_the_engine_lock(gpu_engine):
    x = make_recording(4, 20_000, 2000, 130, seed=1)
    stream = FilterStream(gpu_engine, taps_of("future", 500, 2000 / 130), history=4_000)
    held, release, done = threading.Event(), threading.Event(), []

    def hold():
        with gpu_engine._lock:
            held.set()
            release.wait(60)

    holder = threading.Thread(target=hold)
    holder.start()
    held.wait(10)

    def work():
        done.append(stream.push(x[:, :10_000]).shape)
        done.append(tuple(stream.recent(4_000).shape))
        stream.set_filter(SimpleFilter(taps_of("both", 500, 2000 / 131)))
        done.append(stream.push(x[:, 10_000:]).shape)

    worker = threading.Thread(target=work)
    worker.start()
    worker.join(30)
    finished = not worker.is_alive()
    release.set()
    holder.join()
    worker.join()
    assert finished and len(done) == 3


def fit_errors(monkeypatch, parrm):
    """Run find_period() recording the fit errors of every stage."""
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

    monkeypatch.setattr(PARRM, "_optimise_period_estimate_first_run", first)
    monkeypatch.setattr(PARRM, "_optimise_period_estimate_second_run", second)
    parrm.find_period(random_seed=3)
    monkeypatch.undo()
    return parrm.period, seen


def no_copies(monkeypatch):
    for name in COPIES:
        monkeypatch.setattr(_native.lib, name, lambda *a, _n=name: pytest.fail(f"{_n} called"))


@pytest.mark.parametrize("precision", ["fp64", "fp32"])
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("shape, chunk_bytes", [
    ((6, 40_000), None),          # one channel block, 16-byte rows
    ((5, 40_001), None),          # n_samples x itemsize not a multiple of 16
    ((7, 30_003), 3 * 30_003 * 8),  # blocks of 3 channels (odd rows), unaligned block bases
])
def test_cuda_recording_finds_the_numpy_period_bit_for_bit(gpu_engine, monkeypatch, precision,
                                                           dtype, shape, chunk_bytes):
    import torch

    if chunk_bytes is not None:
        monkeypatch.setattr(_engine, "_SEARCH_CHUNK_BYTES",
                            chunk_bytes // 8 * np.dtype(dtype).itemsize)
    x = make_recording(shape[0], shape[1], 2000, 130, seed=7).astype(dtype)
    host = PARRM(x, 2000, 130, verbose=False, precision=precision)
    want_period, want_errors = fit_errors(monkeypatch, host)
    if chunk_bytes is not None:
        monkeypatch.setattr(_engine, "_SEARCH_CHUNK_BYTES",
                            chunk_bytes // 8 * np.dtype(dtype).itemsize)
    big = torch.zeros((shape[0], shape[1] + 5), dtype=torch.from_numpy(x).dtype, device="cuda")
    big[:, :shape[1]] = torch.from_numpy(x).cuda()
    for data in (torch.from_numpy(x).cuda(), big[:, :shape[1]]):  # dense, and a row-strided view
        dev = PARRM(data, 2000, 130, verbose=False, precision=precision)
        no_copies(monkeypatch)
        if chunk_bytes is not None:
            monkeypatch.setattr(_engine, "_SEARCH_CHUNK_BYTES",
                                chunk_bytes // 8 * np.dtype(dtype).itemsize)
        got_period, got_errors = fit_errors(monkeypatch, dev)
        assert got_period == want_period
        assert len(got_errors) == len(want_errors)
        for (k1, p1, e1), (k2, p2, e2) in zip(got_errors, want_errors):
            assert k1 == k2 and np.array_equal(p1, p2) and np.array_equal(e1, e2)


def test_cuda_recording_filter_and_standard_data(gpu_engine, monkeypatch):
    import torch

    x = make_recording(5, 30_001, 2000, 130, seed=8)
    host = PARRM(x, 2000, 130, verbose=False)
    host.find_period(random_seed=0)
    host.create_filter(filter_half_width=1_000, filter_direction="both")
    want = host.filter_data()
    want_z = host._standard_data
    for data in (torch.from_numpy(x).cuda(), torch.from_numpy(x).cuda()[1:]):
        rows = slice(1, None) if data.shape[0] == 4 else slice(None)
        dev = PARRM(data, 2000, 130, verbose=False)
        no_copies(monkeypatch)
        dev.find_period(random_seed=0)
        dev.create_filter(filter_half_width=1_000, filter_direction="both")
        got = dev.filter_data()
        monkeypatch.undo()
        assert got.is_cuda and got.dtype == torch.float64
        z = dev._standard_data
        assert z.is_cuda and z.dtype == torch.float64
        if rows != slice(None):  # a channel subset: compare with the NumPy twin of those rows
            twin = PARRM(np.ascontiguousarray(x[rows]), 2000, 130, verbose=False)
            twin.find_period(random_seed=0)
            twin.create_filter(filter_half_width=1_000, filter_direction="both")
            host, want, want_z = twin, twin.filter_data(), twin._standard_data
        assert dev.period == host.period
        assert np.array_equal(z.cpu().numpy(), want_z)
        # filter_data(cuda_tensor) and the host pipeline agree to rounding (test_gpu_filter)
        assert np.abs(got.cpu().numpy() - want).max() <= 1e-13 * np.abs(x).max()


def test_cuda_recording_types_and_errors(gpu_engine, monkeypatch):
    import torch

    x = make_recording(3, 20_000, 2000, 130, seed=9)
    parrm = PARRM(torch.from_numpy((x * 100).astype(np.int16)).cuda(), 2000, 130, verbose=False)
    with pytest.raises(TypeError, match="non-floating"):
        parrm.find_period()
    parrm._period = np.float64(2000 / 130 * (1 + 3e-6))
    parrm.create_filter(filter_half_width=500, filter_direction="future")
    got = parrm.filter_data()
    want = gpu_engine.filter_host((x * 100).astype(np.int16), parrm._tap_offsets())
    assert got.is_cuda
    assert np.abs(got.cpu().numpy() - want).max() <= 1e-13 * np.abs(x * 100).max()
    with pytest.raises(TypeError, match="NumPy array"):
        PARRM([[1.0, 2.0]], 2000, 130)
    with pytest.raises(TypeError, match="float64, float32, int16 or int32"):
        PARRM(torch.zeros((2, 100), dtype=torch.float16, device="cuda"), 2000, 130)
    with pytest.raises(TypeError):
        parrm.filter_sweep([{}])
    from pyparrm_b200 import _sharding

    f64 = PARRM(torch.from_numpy(x).cuda(), 2000, 130, verbose=False)
    monkeypatch.setattr(_sharding, "_enabled", True)
    with pytest.raises(NotImplementedError, match="shard"):
        f64.find_period()


def test_frequency_change_recalibrated_from_the_stream(gpu_engine):
    """130 Hz, then 135 Hz from sample 60 000 (fs 2000).  After 10 s of the new frequency the
    stream re-calibrates from its own recent samples and switches: the output matches the
    per-segment gather filter, and the residual artefact on the last 20 000 samples is at least
    5x lower than with the stale taps."""
    x, background = frequency_change_recording()
    history, hw, block = 20_000, 2_000, 500
    cal0 = PARRM(x[:, :history], FS, 130, verbose=False)
    cal0.find_period(random_seed=0)
    cal0.create_filter(filter_half_width=hw, filter_direction="future")
    stream, stale = cal0.filter_stream(history=history), cal0.filter_stream()
    outs, stale_outs, switch = [], [], None
    for t in range(0, x.shape[1], block):
        outs.append(stream.push(x[:, t:t + block]))
        stale_outs.append(stale.push(x[:, t:t + block]))
        if switch is None and stream.n_pushed >= CHANGE + history:
            cal = PARRM(stream.recent(history), FS, F_NEW, verbose=False)
            cal.find_period(random_seed=0)
            cal.create_filter(filter_half_width=hw, filter_direction="future")
            switch = stream.n_emitted
            stream.set_filter(cal)
    outs.append(stream.close())
    stale_outs.append(stale.close())
    got, old = np.concatenate(outs, 1), np.concatenate(stale_outs, 1)
    true = FS / F_NEW * (1 + DRIFT)
    assert abs(cal.period - true) <= 1e-4 * true, cal.period
    want = np.concatenate([
        gpu_engine.filter_host(x, cal0._tap_offsets(), strategy=GATHER)[:, :switch],
        gpu_engine.filter_host(x, cal._tap_offsets(), strategy=GATHER)[:, switch:]], axis=1)
    assert np.array_equal(got, want)
    tail = slice(x.shape[1] - 20_000, None)
    rms = lambda y: float(np.sqrt(np.mean((y[:, tail] - background[:, tail]) ** 2)))  # noqa: E731
    assert rms(old) >= 5 * rms(got), (rms(old), rms(got))

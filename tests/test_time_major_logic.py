"""Time-major recordings, host side (no GPU): which arrays take the time-major path, the time
windows the filter runs in, ``filter_data(out=...)`` validation and ``parrm_transpose``'s
argument errors."""

import ctypes

import numpy as np
import pytest

from oracle import parrm_oracle as oracle
from pyparrm_b200 import PARRM, _engine, _native, _sharding
from pyparrm_b200._engine import (filter_chunks, time_major_input_ld, time_major_ld,
                                  time_major_span, time_windows, window_step)
from tests.oracle_engine import OracleEngine

byte_bounds = getattr(np.lib, "array_utils", np).byte_bounds


# ---------------------------------------------------------------------------------------------
# layout classification
def test_time_major_classification():
    a = np.zeros((1000, 6))
    assert time_major_ld(a) is None                       # C order
    assert time_major_ld(np.zeros((6, 1000))) is None
    assert time_major_ld(a.T) == 6                        # mm.T
    assert time_major_ld(a[:, 1:5].T) == 6                # channel subset: offset base, ld > C
    assert time_major_ld(a[:, 5:6].T) == 6                # one channel of six: (1, T)
    assert time_major_ld(a[10:20].T) == 6                 # a time range
    assert time_major_ld(np.asfortranarray(np.zeros((6, 1000)))) == 6
    assert time_major_ld(a.astype(np.int16).T) == 6
    assert time_major_ld(a[::3].T) == 18                  # every third frame: rows 18 apart
    # rejected: strided channels, negative strides, byte-swapped, wrong rank, not an array
    assert time_major_ld(a[:, ::2].T) is None
    assert time_major_ld(a[::-1].T) is None
    assert time_major_ld(a[:, ::-1].T) is None
    assert time_major_ld(a.astype(a.dtype.newbyteorder()).T) is None
    assert time_major_ld(np.zeros(5)) is None
    assert time_major_ld(a.tolist()) is None
    # (C, 1) and (1, T) shapes NumPy already calls C-contiguous keep the C-order path
    assert np.zeros((1, 6)).T.flags.c_contiguous and time_major_ld(np.zeros((1, 6)).T) is None
    assert time_major_ld(np.zeros((1000, 1)).T) is None
    assert time_major_ld(np.zeros((0, 6)).T) is None


# ---------------------------------------------------------------------------------------------
# time windows
TAP_SETS = {d: oracle.tap_offsets(2000 / 130 * (1 + 3e-6), 2000 / 130 / 50, 200, 0, d)
            for d in ("future", "past", "both")}


@pytest.mark.parametrize("direction", list(TAP_SETS))
@pytest.mark.parametrize("n_samples", [1, 7, 3_200, 50_001, 1_000_000])
@pytest.mark.parametrize("n_chans", [1, 3, 384])
def test_windows_cover_once_with_clipped_halos(direction, n_samples, n_chans):
    taps = TAP_SETS[direction]
    w_lo, w_hi = min(int(taps[0]), 0), max(int(taps[-1]), 0)
    span = w_hi - w_lo
    step = window_step(span, n_chans * 2, n_chans * 8)
    assert step >= 16 * span
    windows = time_windows(n_samples, w_lo, w_hi, step)
    assert windows[0][0] == 0 and windows[-1][1] == n_samples
    for (t0, t1, x0, x1), nxt in zip(windows, windows[1:] + [None]):
        assert t0 < t1 and (nxt is None or nxt[0] == t1)
        # every in-range sample the outputs read, and no more: the halo clipped at both ends
        assert x0 == max(0, t0 - w_hi) and x1 == min(n_samples, t1 - w_lo)
        assert 0 <= x0 <= t0 and t1 <= x1 <= n_samples
        need = [t - w for t in (t0, t1 - 1) for w in taps if 0 <= t - w < n_samples]
        assert all(x0 <= s < x1 for s in need)
        # halo at most 1/16 of a window
        assert (x1 - x0) - (t1 - t0) <= step / 16


def test_window_step_takes_chunk_bytes_or_sixteen_spans(monkeypatch):
    monkeypatch.setattr(_engine, "_CHUNK_BYTES", 32 << 20)
    # cfg4 share: int16 rows of 48 channels up, float64 device buffers of 48 channels
    assert window_step(2311, 48 * 2, 48 * 8) == (32 << 20) // (48 * 8)
    assert window_step(2311, 384 * 2, 384 * 8) == 16 * 2311   # cfg4: the halo rule decides
    assert window_step(0, 8, 8) == (32 << 20) // 8
    # the upload decides when the base's rows are wider than the device buffers
    assert window_step(10, 385 * 4, 2 * 8) == (32 << 20) // (385 * 4)
    monkeypatch.setattr(_engine, "_CHUNK_BYTES", 1)
    assert window_step(0, 5 * 8, 5 * 8) == 1


@pytest.mark.parametrize("n_chans, ld", [(1, 16), (1, 385), (5, 385), (7, 385), (24, 385),
                                         (48, 384), (384, 385)])
@pytest.mark.parametrize("dtype", [np.int16, np.float32])
def test_window_bytes_are_bounded_for_narrow_subsets_of_wide_rows(n_chans, ld, dtype):
    """A window's upload is rows of the base, ``ld`` elements per sample whatever ``C`` is: the
    window length is set by those bytes, so neither the upload nor the ring and the staging
    sized from it exceed about ``_CHUNK_BYTES`` (plus the halo) for a narrow subset of wide
    rows.  Subsets more than ``_TIME_MAJOR_MAX_WIDTH`` times narrower than their rows are not
    read as rows at all."""
    es = np.dtype(dtype).itemsize
    base = np.zeros((9_000, ld), dtype=dtype)
    view = base[:, ld - n_chans:].T
    assert time_major_ld(view) == ld
    assert _engine._TIME_MAJOR_MAX_WIDTH == 64
    if ld > _engine._TIME_MAJOR_MAX_WIDTH * n_chans:
        assert time_major_input_ld(view) is None       # host copy of the channels asked for
        return
    assert time_major_input_ld(view) == ld
    taps = TAP_SETS["past"]
    w_lo, w_hi = min(int(taps[0]), 0), max(int(taps[-1]), 0)
    n_samples = 9_000_000
    for es_c in (4, 8):
        chunks = filter_chunks(n_chans, n_samples, w_lo, w_hi, es, 4, es_c, in_ld=ld,
                               windowed=True)
        assert chunks[0][2] == 0 and chunks[-1][3] == n_samples
        span = w_hi - w_lo
        assert 16 * span * max(ld * es, n_chans * es_c) < _engine._CHUNK_BYTES  # chunk decides
        for c0, c1, t0, t1, x0, x1 in chunks:
            assert (c0, c1) == (0, n_chans)
            up = time_major_span(ld, n_chans, x0, x1, es)[1]
            assert up <= _engine._CHUNK_BYTES + span * ld * es, (up, _engine._CHUNK_BYTES)
            assert n_chans * (x1 - x0) * es_c <= _engine._CHUNK_BYTES + span * n_chans * es_c


def test_default_chunks_are_unchanged():
    """C-order recordings without ``out=``: blocks of whole rows, or one-row time windows."""
    assert filter_chunks(64, 1_200_000, -2000, 2000, 8, 8, 8) == [
        (c0, min(c0 + 3, 64), 0, 1_200_000, 0, 1_200_000) for c0 in range(0, 64, 3)]
    chunks = filter_chunks(2, 9_000_000, -2311, 0, 8, 8, 8)
    step = (32 << 20) // 8
    assert chunks == [(c, c + 1) + w for c in range(2)
                      for w in time_windows(9_000_000, -2311, 0, step)]


@pytest.mark.parametrize("dtype", [np.int16, np.float32, np.float64])
def test_upload_range_stays_inside_the_view(dtype):
    """The bytes a window uploads are rows of the base ending at the view's last channel: never
    past the last byte the view spans (a subset at the end of a mapped file would fault)."""
    base = np.zeros((997, 386), dtype=dtype)
    for lo, hi in ((0, 386), (1, 386), (0, 384), (5, 6), (385, 386)):
        view = base[:, lo:hi].T
        ld = time_major_ld(view)
        first, last = byte_bounds(view)
        assert view.ctypes.data == first
        for x0, x1 in ((0, 997), (0, 1), (996, 997), (100, 731)):
            off, nbytes = time_major_span(ld, view.shape[0], x0, x1, view.itemsize)
            assert first <= first + off and first + off + nbytes <= last
            got = np.frombuffer(base, dtype=np.uint8)[first - base.ctypes.data + off:][:nbytes]
            rows = got.view(dtype)
            # the window's samples are where a [x1 - x0, ld] reading puts them
            idx = np.arange(x1 - x0)[:, None] * ld + np.arange(view.shape[0])[None, :]
            assert idx.max() < rows.size
        off, nbytes = time_major_span(ld, view.shape[0], 0, 997, view.itemsize)
        assert first + off + nbytes == last   # the whole view ends exactly at its last byte


# ---------------------------------------------------------------------------------------------
# filter_data(out=...) validation through a stand-in engine that accepts `out`
class OutEngine(OracleEngine):
    def __init__(self):
        super().__init__()
        self.calls = []

    def filter_host(self, data, taps, precision="fp64", strategy=None, out_dtype=None, out=None):
        result = super().filter_host(data, taps, precision, strategy, out_dtype)
        self.calls.append(out is not None)
        if out is None:
            return result
        out[...] = result
        return out


@pytest.fixture()
def out_engine():
    engine = OutEngine()
    _engine.set_engine(engine)
    yield engine
    _engine.set_engine(None)


def make_parrm(data):
    parrm = PARRM(data, 2000, 130, verbose=False)
    parrm._period = np.float64(2000 / 130)
    parrm.create_filter(filter_half_width=100, filter_direction="both")
    return parrm


def test_out_fills_c_order_and_time_major_arrays(out_engine):
    rng = np.random.default_rng(0)
    base = rng.standard_normal((2_000, 5))
    parrm = make_parrm(base.T)
    want = parrm.filter_data()
    assert out_engine.calls == [False]   # `out` only reaches the engine when given
    for out in (np.empty((5, 2_000)), np.empty((2_000, 5)).T, np.empty((2_000, 7))[:, 1:6].T,
                np.empty((5, 2_000), np.float32)):
        got = parrm.filter_data(out=out)
        assert got is out and parrm.filtered_data is out
        assert np.allclose(got, want, rtol=1e-6 if out.dtype == np.float32 else 0, atol=1e-6)
    got = parrm.filter_data(out=np.empty((5, 2_000), np.float32), out_dtype=np.float32)
    assert got.dtype == np.float32


def test_out_validation(out_engine, monkeypatch):
    data = np.random.default_rng(1).standard_normal((3, 1_000))
    parrm = make_parrm(data)
    with pytest.raises(ValueError, match="shape"):
        parrm.filter_data(out=np.empty((3, 999)))
    with pytest.raises(ValueError, match="shape"):
        parrm.filter_data(out=np.empty((1_000, 3)))
    for dtype in (np.int16, np.float16, np.complex128, np.dtype(">f8")):
        with pytest.raises(TypeError, match="float64 or float32"):
            parrm.filter_data(out=np.empty((3, 1_000), dtype))
    with pytest.raises(TypeError, match="NumPy array"):
        parrm.filter_data(out=[[0.0] * 1_000] * 3)
    with pytest.raises(TypeError, match="out_dtype"):
        parrm.filter_data(out=np.empty((3, 1_000)), out_dtype=np.float32)
    ro = np.empty((3, 1_000))
    ro.flags.writeable = False
    with pytest.raises(ValueError, match="writeable"):
        parrm.filter_data(out=ro)
    with pytest.raises(ValueError, match="share memory"):
        parrm.filter_data(out=data)
    frames = np.zeros((1_000, 6))
    with pytest.raises(ValueError, match="share memory"):   # channels of the same frames
        parrm.filter_data(frames[:, :3].T, out=frames[:, 3:].T)
    with pytest.raises(ValueError, match="C-contiguous or time-major"):
        parrm.filter_data(out=np.empty((3, 2_000))[:, ::2])
    assert out_engine.calls == []
    monkeypatch.setattr(_sharding, "active", lambda: True)
    with pytest.raises(NotImplementedError, match="out"):
        parrm.filter_data(out=np.empty((3, 1_000)))


def test_out_with_a_cuda_tensor_is_refused(out_engine):
    class FakeCuda:   # what PARRM's tensor check looks at, no torch device needed
        __module__ = "torch.fake"
        is_cuda = True
        ndim = 2

        def dim(self):
            return 2

    parrm = make_parrm(np.zeros((2, 500)))
    with pytest.raises(TypeError, match="`out` applies to NumPy"):
        parrm.filter_data(FakeCuda(), out=np.empty((2, 500)))


# ---------------------------------------------------------------------------------------------
# parrm_transpose argument errors (checked before anything is enqueued: no device needed)
def test_transpose_argument_errors():
    lib = _native.lib
    fake = ctypes.c_void_p(4096)
    cases = [
        ((None, 0, 4, 4, 4, fake, 0, 4), "null"),
        ((fake, 0, 4, 4, 4, None, 0, 4), "null"),
        ((fake, 7, 4, 4, 4, fake, 0, 4), "unknown source"),
        ((fake, 0, 4, 4, 4, fake, 9, 4), "unknown destination"),
        ((fake, 2, 4, 4, 4, fake, 3, 4), "unsupported type pair"),    # int16 -> int32
        ((fake, 0, 4, 4, 4, fake, 2, 4), "unsupported type pair"),    # float64 -> int16
        ((fake, 1, 4, 4, 3, fake, 1, 4), "src_ld"),
        ((fake, 1, 4, 4, 4, fake, 1, 3), "dst_ld"),
        ((fake, 1, -1, 4, 4, fake, 1, 4), "negative"),
    ]
    for args, msg in cases:
        assert lib.parrm_transpose(*args, None) == 1, msg
        assert msg in _native.last_error(), (msg, _native.last_error())
    assert lib.parrm_transpose(fake, 2, 0, 4, 4, fake, 0, 0, None) == 0   # nothing to do
    # an unsupported pair is refused whatever the shape, empty ones included
    for rows, cols in ((0, 4), (4, 0), (0, 0)):
        assert lib.parrm_transpose(fake, 2, rows, cols, 4, fake, 3, 4, None) == 1
        assert "unsupported type pair" in _native.last_error()
    for fn in (lib.parrm_copy_d2h_2d_async, lib.parrm_copy_h2d_2d_async):
        assert fn(None, 8, fake, 8, 8, 2, None) == 1 and "null" in _native.last_error()
        assert fn(fake, 4, fake, 8, 8, 2, None) == 1 and "pitch" in _native.last_error()
        assert fn(None, 8, None, 8, 0, 2, None) == 0

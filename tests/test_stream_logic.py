"""Host logic of the streaming filter (``PARRM.filter_stream``) on a CPU stand-in engine, and the
argument checks of its C entry points on a host without a GPU.

The stand-in keeps the tail of the recording a push can still read (what the device ring
holds) and filters the window of each push with the oracle, so every output is computed from
the samples a real push has at hand; concatenated, the pushes must equal the oracle on the
whole recording bit for bit.
"""

import ctypes
from types import SimpleNamespace

import numpy as np
import pytest

from oracle import parrm_oracle as oracle
from pyparrm_b200 import PARRM, _engine, _native, _sharding
from pyparrm_b200._stream import FilterStream, output_range
from tests.oracle_engine import OracleEngine

PERIOD = 2000 / 130 * (1 + 3e-6)
NO_FILTER = "The filter has not yet been created"


class StreamOracleEngine(OracleEngine):
    """``OracleEngine`` plus the two stream entry points of ``DeviceEngine``."""

    def __init__(self):
        super().__init__()
        self.pushes = []  # (pos, n, close) of every push that reached the engine

    def stream_open(self, taps, max_chunk, precision="fp64"):
        taps = np.array(taps, dtype=np.int32)
        return SimpleNamespace(taps=taps, max_chunk=max_chunk, latency=max(0, -int(taps[0])),
                               w_hi=max(0, int(taps[-1])), tail=None, tail_t0=0, n_chans=None,
                               device=None)

    def stream_push(self, st, block, pos, close, out_dtype=None, graphs=True):
        if block is None:
            block = np.zeros((st.n_chans, 0))
        block = np.asarray(block, dtype=np.float64)
        n = block.shape[1]
        assert n <= st.max_chunk
        self.pushes.append((pos, n, close))
        st.n_chans = block.shape[0]
        x = block if st.tail is None else np.concatenate([st.tail, block], axis=1)
        lo, hi = output_range(pos, n, st.latency, close)
        win0 = max(0, lo - st.w_hi)            # oldest sample these outputs read
        assert win0 >= st.tail_t0
        window = x[:, win0 - st.tail_t0:]       # samples [win0, pos + n)
        with np.errstate(invalid="ignore"):
            y = oracle.apply_filter_direct(window, st.taps)[:, lo - win0:hi - win0]
        y[~np.isfinite(y)] = 0.0
        keep = max(0, pos + n - st.latency - st.w_hi)  # what the next push can still read
        st.tail, st.tail_t0 = x[:, keep - st.tail_t0:], keep
        return y.astype(np.float64 if out_dtype is None else out_dtype)


@pytest.fixture()
def stream_engine():
    engine = StreamOracleEngine()
    _engine.set_engine(engine)
    yield engine
    _engine.set_engine(None)


def make_parrm(data, direction="both", hw=300):
    parrm = PARRM(data, 2000, 130, verbose=False)
    parrm._period = np.float64(PERIOD)
    parrm.create_filter(filter_half_width=hw, filter_direction=direction)
    return parrm


def stream_all(stream, x, sizes):
    outs, t = [], 0
    for n in sizes:
        outs.append(stream.push(x[:, t:t + n]))
        t += n
    assert t == x.shape[1]
    outs.append(stream.close())
    return np.concatenate(outs, axis=1)


def random_sizes(rng, total, span):
    sizes = []
    pool = [1, 2, 3, 7, 13, 101, span, span - 1, span + 1, 997]
    while sum(sizes) < total:
        sizes.append(int(rng.choice(pool)) if rng.random() < 0.7 else int(rng.integers(1, 3 * span)))
    sizes[-1] -= sum(sizes) - total
    return [s for s in sizes if s > 0]


@pytest.mark.parametrize("direction", ["both", "past", "future"])
def test_pushes_concatenate_to_the_whole_recording(stream_engine, direction):
    rng = np.random.default_rng(len(direction))
    x = rng.standard_normal((3, 9_000)) * 5 + 20
    parrm = make_parrm(x, direction)
    taps = parrm._tap_offsets()
    want = oracle.apply_filter_direct(x, taps)
    span = max(int(taps[-1]), 0) - min(int(taps[0]), 0)
    for seed in range(3):
        sizes = random_sizes(np.random.default_rng(seed), x.shape[1], span)
        stream = parrm.filter_stream()
        got = stream_all(stream, x, sizes)
        assert np.array_equal(got, want), (direction, seed)
        assert stream.n_pushed == stream.n_emitted == x.shape[1]
    # every push returns exactly the outputs that are final: t < pushed - latency
    stream = parrm.filter_stream()
    pushed = 0
    for n in (1, 5, stream.latency + 3, 1, 250):
        y = stream.push(x[:, pushed:pushed + n])
        before = max(0, pushed - stream.latency)
        pushed += n
        assert y.shape == (3, max(before, pushed - stream.latency) - before)
    assert stream.close().shape == (3, min(pushed, stream.latency))


def test_latency_follows_the_taps_not_the_name(stream_engine):
    x = np.zeros((1, 5000))
    hw = 300
    got = {d: make_parrm(x, d, hw).filter_stream().latency for d in ("both", "past", "future")}
    assert got["future"] == 0                       # y[t] reads x[t - w], w > 0: causal
    for d in ("both", "past"):
        taps = make_parrm(x, d, hw)._tap_offsets()
        assert got[d] == -int(taps[0]) and 0 < got[d] <= hw


@pytest.mark.parametrize("direction", ["both", "past"])
def test_stream_shorter_than_the_latency_comes_out_at_close(stream_engine, direction):
    x = np.random.default_rng(3).standard_normal((2, 40))
    parrm = make_parrm(np.zeros((2, 5000)), direction)
    stream = parrm.filter_stream()
    assert stream.latency > x.shape[1]
    for piece in np.array_split(x, 4, axis=1):
        assert stream.push(piece).shape == (2, 0)
    tail = stream.close()
    assert np.array_equal(tail, oracle.apply_filter_direct(x, parrm._tap_offsets()))


def test_taps_are_a_snapshot(stream_engine):
    x = np.random.default_rng(4).standard_normal((2, 3000))
    parrm = make_parrm(x, "past")
    taps = parrm._tap_offsets()
    stream = parrm.filter_stream(out_dtype=np.float32)
    parrm.create_filter(filter_half_width=100, filter_direction="future")
    assert np.array_equal(stream.taps, taps)
    got = stream_all(stream, x, [700, 1300, 1000])
    assert got.dtype == np.float32
    assert np.array_equal(got, oracle.apply_filter_direct(x, taps).astype(np.float32))


def test_max_chunk_splits_long_pushes(stream_engine):
    x = np.random.default_rng(5).standard_normal((2, 2000))
    parrm = make_parrm(x, "both", hw=100)
    stream = parrm.filter_stream(max_chunk=7)
    got = stream_all(stream, x, [1, 100, 1899])
    assert np.array_equal(got, oracle.apply_filter_direct(x, parrm._tap_offsets()))
    assert max(n for _, n, _ in stream_engine.pushes) == 7
    assert sum(n for _, n, _ in stream_engine.pushes) == 2000
    positions = [p for p, _, _ in stream_engine.pushes]
    assert positions == sorted(positions)


def test_non_finite_samples_across_block_boundaries(stream_engine):
    rng = np.random.default_rng(6)
    x = rng.standard_normal((2, 4000))
    x[0, 999], x[0, 1000], x[1, 1001] = np.nan, np.inf, -np.inf
    parrm = make_parrm(x, "both", hw=200)
    taps = parrm._tap_offsets()
    with np.errstate(invalid="ignore"):
        want = oracle.apply_filter_direct(x, taps)
    want[~np.isfinite(want)] = 0.0
    got = stream_all(parrm.filter_stream(), x, [1000, 1, 2999])
    assert np.array_equal(got, want)


def test_error_paths(stream_engine, monkeypatch):
    x = np.zeros((3, 5000))
    parrm = PARRM(x, 2000, 130, verbose=False)
    parrm._period = np.float64(PERIOD)
    with pytest.raises(ValueError, match=NO_FILTER):
        parrm.filter_stream()
    with pytest.raises(ValueError, match=NO_FILTER):
        parrm.filter_data()
    parrm.create_filter(filter_half_width=300)
    with pytest.raises(TypeError, match="max_chunk"):
        parrm.filter_stream(max_chunk=2.5)
    with pytest.raises(ValueError, match="max_chunk"):
        parrm.filter_stream(max_chunk=0)
    with pytest.raises(TypeError, match="out_dtype"):
        parrm.filter_stream(out_dtype=np.int16)
    with pytest.raises(TypeError):
        parrm.filter_stream(1024)  # keyword-only
    monkeypatch.setattr(_sharding, "_enabled", True)
    with pytest.raises(NotImplementedError, match="shard"):
        parrm.filter_stream()
    monkeypatch.setattr(_sharding, "_enabled", False)

    stream = parrm.filter_stream()
    with pytest.raises(TypeError, match="NumPy array or a CUDA tensor"):
        stream.push([[1.0, 2.0]])
    with pytest.raises(ValueError, match="2D"):
        stream.push(np.zeros(10))
    empty = stream.push(np.zeros((3, 0)))
    assert empty.shape == (3, 0) and empty.dtype == np.float64
    assert stream_engine.pushes == []  # a zero-length push never reaches the engine
    stream.push(np.ones((3, 10), dtype=np.int16))
    with pytest.raises(ValueError, match="3"):
        stream.push(np.zeros((4, 10)))
    assert stream.push(np.zeros((3, 0))).shape == (3, 0)
    assert stream.close().shape == (3, 10)
    with pytest.raises(RuntimeError, match="closed"):
        stream.push(np.zeros((3, 10)))
    with pytest.raises(RuntimeError, match="closed"):
        stream.close()
    # nothing pushed: close gives nothing
    assert parrm.filter_stream().close().shape == (0, 0)


def test_c_entry_points_report_argument_errors():
    """The checks run before any CUDA call, so they hold on a host without a GPU."""
    lib = _native.lib
    taps = np.array([-5, -2, 3, 9], dtype=np.int32)
    ptr = ctypes.c_void_p(taps.ctypes.data)
    # ring: span 14 + max_chunk 100 samples per channel
    assert lib.parrm_stream_ring_bytes(3, ptr, 4, 100, _native.F64) == 3 * 114 * 8
    assert lib.parrm_stream_ring_bytes(3, ptr, 4, 100, _native.F32) == 3 * 114 * 4
    bad = np.array([3, 1], dtype=np.int32)
    assert lib.parrm_stream_ring_bytes(3, ctypes.c_void_p(bad.ctypes.data), 2, 100, 0) == 0
    assert "ascending" in _native.last_error()
    assert lib.parrm_stream_ring_bytes(3, ptr, 4, 0, 0) == 0

    def push(**kw):
        a = dict(ring=None, n_chans=3, max_chunk=100, taps=None, n_taps=4, w_min=-5, w_max=9,
                 block=None, block_type=_native.I16, ld_block=50, n=50, out=None,
                 out_type=_native.F32, ld_out=50, pos=0, d_pos=None, close=0, dtype=_native.F64)
        a.update(kw)
        return lib.parrm_stream_push(*a.values(), None)

    assert push(n=101) == 1 and "longer than the ring" in _native.last_error()
    assert push(pos=-1) == 1 and "backwards" in _native.last_error()
    assert push(dtype=7) == 1 and "dtype" in _native.last_error()
    assert push(block_type=9) == 1 and "storage type" in _native.last_error()
    assert push(out_type=_native.I16) == 1 and "output type" in _native.last_error()
    assert push(n_chans=0) == 1 and "channels" in _native.last_error()
    assert push(w_min=10) == 1 and "tap list" in _native.last_error()
    assert push() == 1 and "null ring" in _native.last_error()


def test_output_range_bookkeeping():
    assert output_range(0, 10, 0, False) == (0, 10)
    assert output_range(0, 10, 25, False) == (0, 0)
    assert output_range(10, 10, 25, False) == (0, 0)
    assert output_range(20, 10, 25, False) == (0, 5)
    assert output_range(30, 10, 25, False) == (5, 15)
    assert output_range(40, 0, 25, True) == (15, 40)
    assert output_range(10, 0, 25, True) == (0, 10)
    with pytest.raises(ValueError, match="ascending"):
        FilterStream(StreamOracleEngine(), [3, 1])

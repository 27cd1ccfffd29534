"""Re-calibrating an open stream (``filter_stream(history=...)``, ``recent()``, ``set_filter()``)
on a CPU stand-in engine, and the argument checks of the C entry points behind it on a host
without a GPU.

The stand-in models the device ring: it keeps exactly the last ``ring_len`` samples, asserts
the ring invariant of ``parrm_stream_push_at`` on every push, and filters each push's window
with the oracle.  Pushed across tap switches, the outputs must concatenate to the oracle on the
whole recording with each tap set over its own range of outputs, bit for bit.
"""

import threading
from types import SimpleNamespace

import numpy as np
import pytest

from oracle import parrm_oracle as oracle
from pyparrm_b200 import PARRM, _engine, _native
from pyparrm_b200._stream import output_range
from tests.oracle_engine import OracleEngine

PERIOD = 2000 / 130 * (1 + 3e-6)
NO_FILTER = "The filter has not yet been created"


class RingOracleEngine(OracleEngine):
    """``OracleEngine`` plus the stream entry points of ``DeviceEngine``, with a ring of
    ``max(span, history) + max_chunk`` samples per channel as the device keeps it."""

    def __init__(self):
        super().__init__()
        self.pushes = []     # (pos, n, close, emitted keyword or None)
        self.opens = []      # keywords stream_open was called with

    def stream_open(self, taps, max_chunk, precision="fp64", **kw):
        self.opens.append(kw)
        taps = np.array(taps, dtype=np.int32)
        span = max(int(taps[-1]), 0) - min(int(taps[0]), 0)
        return SimpleNamespace(taps=taps, max_chunk=max_chunk, latency=max(0, -int(taps[0])),
                               ring_len=max(span, kw.get("history", 0)) + max_chunk,
                               ring=None, ring_t0=0, n_chans=None, device=None)

    def stream_retune(self, st, taps):
        st.taps = np.array(taps, dtype=np.int32)
        st.latency = max(0, -int(st.taps[0]))

    def stream_recent(self, st, n, pos):
        assert st.ring_t0 + st.ring.shape[1] == pos
        return st.ring[:, st.ring.shape[1] - n:].copy()

    def stream_push(self, st, block, pos, close, out_dtype=None, graphs=False, emitted=None):
        if block is None:
            block = np.zeros((st.n_chans, 0))
        block = np.asarray(block, dtype=np.float64)
        n = block.shape[1]
        assert n <= st.max_chunk
        self.pushes.append((pos, n, close, emitted))
        st.n_chans = block.shape[0]
        x = block if st.ring is None else np.concatenate([st.ring, block], axis=1)
        lo, hi = output_range(pos, n, st.latency, close, emitted)
        assert 0 <= lo <= pos
        win0 = max(0, lo - max(0, int(st.taps[-1])))  # oldest sample these outputs read
        assert pos + n - win0 <= st.ring_len            # the ring invariant of push_at
        assert win0 >= st.ring_t0
        window = x[:, win0 - st.ring_t0:]                # samples [win0, pos + n)
        with np.errstate(invalid="ignore"):
            y = oracle.apply_filter_direct(window, st.taps)[:, lo - win0:hi - win0]
        y[~np.isfinite(y)] = 0.0
        keep = max(0, pos + n - st.ring_len)             # the ring after this push
        st.ring, st.ring_t0 = x[:, keep - st.ring_t0:], keep
        return y.astype(np.float64 if out_dtype is None else out_dtype)


@pytest.fixture()
def ring_engine():
    engine = RingOracleEngine()
    _engine.set_engine(engine)
    yield engine
    _engine.set_engine(None)


def make_parrm(data, direction="both", hw=300, period=PERIOD):
    parrm = PARRM(data, 2000, 130, verbose=False)
    parrm._period = np.float64(period)
    parrm.create_filter(filter_half_width=hw, filter_direction=direction)
    return parrm


def stream_with_switches(stream, x, sizes, switches):
    """Push ``x`` in blocks of ``sizes``; before push ``i`` in ``switches`` (``len(sizes)``:
    before ``close()``) switch to ``switches[i]``.  Returns the concatenated outputs and the
    ``[(switch point, taps)]`` segments, checking that ``n_emitted`` always equals the columns
    returned."""
    segments = [(0, stream.taps)]
    outs, t, cols = [], 0, 0
    for i, n in enumerate(sizes + [None]):
        if i in switches:
            stream.set_filter(switches[i])
            segments.append((stream.n_emitted, stream.taps))
        y = stream.close() if n is None else stream.push(x[:, t:t + n])
        t += 0 if n is None else n
        cols += y.shape[1]
        outs.append(y)
        assert stream.n_emitted == cols and stream.n_pushed == t
    assert t == x.shape[1] and cols == x.shape[1]
    return np.concatenate(outs, axis=1), segments


def per_segment(x, segments):
    """The contract: filter_data over the whole recording with taps_k on [s_k, s_k+1)."""
    bounds = [s for s, _ in segments[1:]] + [x.shape[1]]
    parts, s0 = [], 0
    for (s, taps), s1 in zip(segments, bounds):
        assert s == s0
        parts.append(oracle.apply_filter_direct(x, taps)[:, s:s1])
        s0 = s1
    return np.concatenate(parts, axis=1)


def seeded_sizes(rng, total):
    sizes = []
    while sum(sizes) < total:
        sizes.append(int(rng.choice([1, 7, 13, 101, 299, 300, 301, 997, 2500])))
    sizes[-1] -= sum(sizes) - total
    return [s for s in sizes if s > 0]


@pytest.mark.parametrize("old, new", [("future", "both"),    # latency grows
                                      ("past", "future"),    # latency shrinks
                                      ("both", "both")])     # latency equal
def test_one_switch_matches_the_per_segment_filter(ring_engine, old, new):
    rng = np.random.default_rng(len(old) * 7 + len(new))
    x = rng.standard_normal((3, 9_000)) * 5 + 20
    first, second = make_parrm(x, old), make_parrm(x, new, hw=250, period=PERIOD * 1.01)
    for seed in range(3):
        r = np.random.default_rng(seed)
        sizes = seeded_sizes(r, x.shape[1])
        at = int(r.integers(1, len(sizes)))
        stream = first.filter_stream(history=1_000)
        got, segments = stream_with_switches(stream, x, sizes, {at: second})
        assert np.array_equal(got, per_segment(x, segments)), (seed, at)
        assert stream.latency == max(0, -int(second._tap_offsets()[0]))
        emitted = [e for _, _, _, e in ring_engine.pushes]
        ring_engine.pushes.clear()
        assert emitted[:at] == [None] * at  # before the switch the engine is called as before
        assert None not in emitted[at:]


def test_several_switches_before_the_first_push_and_before_close(ring_engine):
    rng = np.random.default_rng(11)
    x = rng.standard_normal((2, 12_000))
    parrms = [make_parrm(x, d, hw, PERIOD * f) for d, hw, f in
              (("both", 300, 1.0), ("future", 200, 0.99), ("past", 350, 1.02),
               ("both", 150, 1.0), ("future", 400, 1.01))]
    for seed in range(4):
        r = np.random.default_rng(100 + seed)
        sizes = seeded_sizes(r, x.shape[1])
        points = sorted(r.choice(np.arange(1, len(sizes)), 2, replace=False).tolist())
        switches = {0: parrms[1], points[0]: parrms[2], points[1]: parrms[3],
                    len(sizes): parrms[4]}
        stream = parrms[0].filter_stream(history=1_200, max_chunk=1_000)
        got, segments = stream_with_switches(stream, x, sizes, switches)
        assert len(segments) == 5 and segments[1][0] == 0
        assert np.array_equal(got, per_segment(x, segments)), seed
    assert max(n for _, n, _, _ in ring_engine.pushes) == 1_000


def test_float32_results_across_a_switch(ring_engine):
    x = np.random.default_rng(3).standard_normal((2, 5_000))
    a, b = make_parrm(x, "past"), make_parrm(x, "future", hw=200)
    stream = a.filter_stream(history=800, out_dtype=np.float32)
    got, segments = stream_with_switches(stream, x, [1_000, 1_500, 2_500], {2: b})
    assert got.dtype == np.float32
    assert np.array_equal(got, per_segment(x, segments).astype(np.float32))


def test_history_and_no_switch_call_the_engine_as_before(ring_engine):
    x = np.random.default_rng(4).standard_normal((2, 3_000))
    parrm = make_parrm(x)
    plain = parrm.filter_stream()
    kept = parrm.filter_stream(history=5_000)
    assert ring_engine.opens == [{}, {"history": 5_000}]
    span = plain.ring_len - plain.max_chunk
    assert kept.ring_len == 5_000 + kept.max_chunk and span < 5_000
    for stream in (plain, kept):
        got, _ = stream_with_switches(stream, x, [1_000, 2_000], {})
        assert np.array_equal(got, oracle.apply_filter_direct(x, parrm._tap_offsets()))
    assert all(e is None for _, _, _, e in ring_engine.pushes)


def test_recent_returns_the_last_samples(ring_engine):
    x = np.random.default_rng(5).standard_normal((3, 6_000))
    parrm = make_parrm(x, hw=100)
    stream = parrm.filter_stream(history=2_500, max_chunk=700)
    with pytest.raises(ValueError, match="history"):
        stream.recent(1)                     # nothing pushed yet
    t = 0
    for n in (1_000, 3_000, 1, 1_999):
        stream.push(x[:, t:t + n])
        t += n
        for k in (1, min(t, 2_500)):
            assert np.array_equal(stream.recent(k), x[:, t - k:t])
    with pytest.raises(ValueError, match="history = 2500"):
        stream.recent(2_501)
    small = parrm.filter_stream(history=50)
    small.push(x[:, :40])
    with pytest.raises(ValueError, match="history"):
        small.recent(41)                     # more than was pushed
    with pytest.raises(ValueError, match="history"):
        small.recent(0)
    with pytest.raises(TypeError):
        small.recent(2.0)
    stream.close()
    with pytest.raises(RuntimeError, match="closed"):
        stream.recent(10)


def test_set_filter_validation(ring_engine):
    x = np.zeros((3, 5_000))
    parrm = make_parrm(x, "both", hw=300)
    span = parrm.filter_stream().ring_len - (1 << 16)
    unfiltered = PARRM(x, 2000, 130, verbose=False)
    stream = parrm.filter_stream()
    with pytest.raises(ValueError, match=NO_FILTER):
        stream.set_filter(unfiltered)
    wide = make_parrm(x, "both", hw=600)
    with pytest.raises(ValueError, match=r"history=\d+"):
        stream.set_filter(wide)               # its span does not fit the ring
    stream.push(x[:, :2_000])
    assert stream.n_pushed - stream.n_emitted == stream.latency > 250
    # span fits, but the pending outputs reach back further than the ring holds
    late = make_parrm(x, "future", hw=450)
    assert max(0, int(late._tap_offsets()[-1])) + stream.latency > span >= 450
    with pytest.raises(ValueError, match="pending outputs reach back") as err:
        stream.set_filter(late)
    need = int(str(err.value).split("history=")[1].split(")")[0])
    assert np.array_equal(stream.taps, parrm._tap_offsets())  # nothing changed
    roomy = parrm.filter_stream(history=need)
    roomy.push(x[:, :2_000])
    roomy.set_filter(late)                    # the history the message names is enough
    stream.close()
    with pytest.raises(RuntimeError, match="closed"):
        stream.set_filter(parrm)
    with pytest.raises(TypeError, match="history"):
        parrm.filter_stream(history=1.5)
    with pytest.raises(ValueError, match="history"):
        parrm.filter_stream(history=-1)


def test_pushes_do_not_take_the_engine_lock(ring_engine):
    ring_engine._lock = threading.RLock()
    x = np.random.default_rng(6).standard_normal((2, 4_000))
    a, b = make_parrm(x, "future", hw=200), make_parrm(x, "both", hw=200)
    stream = a.filter_stream(history=1_000)
    held, release = threading.Event(), threading.Event()

    def hold():
        with ring_engine._lock:
            held.set()
            release.wait(30)

    holder = threading.Thread(target=hold)
    holder.start()
    held.wait(10)
    done = []

    def work():
        stream.push(x[:, :2_000])
        stream.recent(500)
        stream.set_filter(b)
        done.append(stream.push(x[:, 2_000:]).shape)

    worker = threading.Thread(target=work)
    worker.start()
    worker.join(10)
    finished = not worker.is_alive()
    release.set()
    holder.join()
    worker.join()
    assert finished and done


def test_output_range_with_and_without_emitted():
    assert output_range(30, 10, 25, False) == (5, 15)
    assert output_range(30, 10, 25, False, emitted=5) == (5, 15)     # the same when consistent
    assert output_range(30, 10, 25, False, emitted=0) == (0, 15)     # latency shrank: more than n
    assert output_range(30, 10, 45, False, emitted=5) == (5, 5)      # latency grew: none
    assert output_range(30, 10, 0, False, emitted=12) == (12, 40)
    assert output_range(40, 0, 25, True, emitted=3) == (3, 40)
    assert output_range(0, 10, 0, False, emitted=0) == (0, 10)


def test_c_entry_points_report_argument_errors():
    """The checks run before any CUDA call, so they hold on a host without a GPU."""
    lib = _native.lib

    def push_at(**kw):
        a = dict(ring=None, ring_len=200, n_chans=3, taps=None, n_taps=4, w_min=-5, w_max=9,
                 block=None, block_type=_native.I16, ld_block=50, n=50, out=None,
                 out_type=_native.F32, ld_out=100, pos=1_000, out_lo=995, d_hdr=None, close=0,
                 dtype=_native.F64)
        a.update(kw)
        return lib.parrm_stream_push_at(*a.values(), None)

    # reach = pos + n - (out_lo - w_max) = 1000 + 50 - 986 = 64 <= 200: only the null ring fails
    assert push_at() == 1 and "null ring" in _native.last_error()
    assert push_at(ring_len=63) == 1 and "ring" in _native.last_error()
    assert push_at(out_lo=800) == 1 and "more than the ring" in _native.last_error()  # 259
    assert push_at(out_lo=1_001) == 1 and "first output" in _native.last_error()
    assert push_at(out_lo=-1) == 1 and "first output" in _native.last_error()
    assert push_at(n=-1) == 1 and "negative" in _native.last_error()
    assert push_at(pos=-1, out_lo=0) == 1 and "position" in _native.last_error()
    assert push_at(dtype=7) == 1 and "dtype" in _native.last_error()
    assert push_at(w_min=10) == 1 and "tap list" in _native.last_error()
    assert push_at(ring_len=0) == 1 and "ring length" in _native.last_error()

    def window(**kw):
        a = dict(ring=None, ring_len=100, n_chans=3, pos=500, n=60, dst=None, ld_dst=60,
                 dtype=_native.F32)
        a.update(kw)
        return lib.parrm_stream_window(*a.values(), None)

    assert window() == 1 and "null ring" in _native.last_error()
    assert window(n=101) == 1 and "window of 101" in _native.last_error()   # more than the ring
    assert window(pos=50) == 1 and "window of 60" in _native.last_error()   # more than pushed
    assert window(n=0) == 1 and "window" in _native.last_error()
    assert window(dtype=_native.I16) == 1 and "dtype" in _native.last_error()
    assert window(n_chans=0) == 1 and "channels" in _native.last_error()


# ---- end-to-end frequency change: the recording is shared with the GPU test --------------------
FS, F_OLD, F_NEW, CHANGE, DRIFT = 2000, 130, 135, 60_000, 3e-6


def frequency_change_recording(n_chans=4, n_samples=120_000, seed=0):
    """``(x, background)``: white background plus an artefact at 130 Hz for the first
    ``CHANGE`` samples and at 135 Hz after (the stimulation reprogrammed mid-session), both
    periods carrying the synthetic clock mismatch ``DRIFT``."""
    rng = np.random.default_rng(seed)
    background = rng.standard_normal((n_chans, n_samples))
    amps = rng.uniform(2.0, 5.0, n_chans)
    phases = rng.uniform(0.0, 2 * np.pi, 5)
    t = np.arange(n_samples, dtype=np.float64)
    wave = np.zeros(n_samples)
    for freq, sl in ((F_OLD, slice(0, CHANGE)), (F_NEW, slice(CHANGE, None))):
        period = FS / freq * (1 + DRIFT)
        for k in range(1, 6):
            wave[sl] += np.sin(2 * np.pi * k / period * t[sl] + phases[k - 1]) / k
    return background + amps[:, None] * wave, background


def test_frequency_change_margin_with_the_true_periods():
    """What the GPU test relies on: with the true periods, switching the taps after the
    frequency change lowers the residual artefact on the last 20 000 samples at least 5x."""
    x, background = frequency_change_recording()
    hw = 2_000
    taps = {f: oracle.tap_offsets(FS / f * (1 + DRIFT), FS / f * (1 + DRIFT) / 50, hw, 0,
                                  "future") for f in (F_OLD, F_NEW)}
    stale = oracle.apply_filter_direct(x, taps[F_OLD])
    switched = oracle.apply_filter_direct(x, taps[F_NEW])
    tail = slice(x.shape[1] - 20_000, None)
    rms = lambda y: float(np.sqrt(np.mean((y[:, tail] - background[:, tail]) ** 2)))  # noqa: E731
    assert rms(stale) >= 5 * rms(switched), (rms(stale), rms(switched))

"""Streaming filter on the B200: pushes + close are bit-equal to the gather filter on the whole
recording (``filter_host(..., strategy=PLAN_GATHER)``), whatever the block sizes, storage types,
precision, output type, input residency or graph replay."""

import numpy as np
import pytest

from oracle import parrm_oracle as oracle
from pyparrm_b200 import PARRM, _native, get_example_data_paths
from pyparrm_b200._stream import FilterStream
from pyparrm_b200.synthetic import make_recording

pytestmark = pytest.mark.gpu
GATHER = _native.PLAN_GATHER


def rel_err(got, want, scale):
    return float(np.abs(got - want).max() / scale) if got.size else 0.0


def span_of(taps):
    return max(int(taps[-1]), 0) - min(int(taps[0]), 0)


def block_sizes(seed, total, span, max_chunk):
    """Seeded block sizes: 1, primes, exactly the span, longer than max_chunk, random."""
    rng = np.random.default_rng(seed)
    pool = [1, 2, 3, 7, 13, 101, 1009, span, max_chunk + 123]
    sizes = []
    while sum(sizes) < total:
        sizes.append(int(rng.choice(pool)) if rng.random() < 0.7 else int(rng.integers(1, 4000)))
    sizes[-1] -= sum(sizes) - total
    return [s for s in sizes if s > 0]


def run_stream(engine, taps, x, sizes, **kw):
    stream = FilterStream(engine, taps, **kw)
    outs, t = [], 0
    for n in sizes:
        outs.append(stream.push(x[:, t:t + n]))
        t += n
    outs.append(stream.close())
    if hasattr(outs[0], "is_cuda"):
        import torch

        return torch.cat(outs, dim=1)
    return np.concatenate(outs, axis=1)


def check_stream(engine, x, taps, seed, want_ref=None, cols=None, max_chunk=4096):
    got = run_stream(engine, taps, x, block_sizes(seed, x.shape[1], span_of(taps), max_chunk),
                     max_chunk=max_chunk, graphs=False)
    assert np.array_equal(got, engine.filter_host(x, taps, strategy=GATHER))
    scale = np.abs(x).max()
    assert rel_err(got, oracle.apply_filter_direct(x, taps), scale) <= 1e-13
    ok = oracle.in_range_tap_count(x.shape[1], taps) > 0
    assert np.all(got[:, ~ok] == 0)
    if want_ref is not None:
        if cols is not None:
            got, ok = got[:, cols], ok[cols]
        assert rel_err(got[:, ok], want_ref[:, ok], scale) <= 1e-9


@pytest.mark.parametrize("name", ["both", "past", "future"])
def test_synthetic_bit_equal_to_the_whole_recording(golden, gpu_engine, name):
    g = golden("synthetic_2x30000")
    n_chans, n, fs, fa, seed = (int(v) for v in g["recording"])
    data = make_recording(n_chans, n, fs, fa, seed=seed)
    for s in range(3):
        check_stream(gpu_engine, data, g[f"{name}_taps"], s, g[f"{name}_filtered"],
                     g[f"{name}_filtered_cols"])


@pytest.mark.parametrize("which", ["taps", "default_taps"])
def test_example_dbs_bit_equal(golden, gpu_engine, which):
    g = golden("example_dbs")
    data = np.load(get_example_data_paths("example_data"))
    want = g["filtered"] if which == "taps" else g["default_filtered"]
    for s in range(2):
        check_stream(gpu_engine, data, g[which], s, want, max_chunk=2048)


def test_span_wider_than_shared_memory(gpu_engine):
    """An 80 000-sample span: the global-memory kernel reads the ring from L2."""
    rng = np.random.default_rng(1)
    x = rng.standard_normal((2, 200_000))
    taps = oracle.tap_offsets(230.77, 4.6, 40_000, 0, "both")
    assert span_of(taps) * 8 > 200 * 1024
    got = run_stream(gpu_engine, taps, x, [1, 30_011, 65_536, 7, 41_000, 63_445],
                     graphs=False)
    assert np.array_equal(got, gpu_engine.filter_host(x, taps, strategy=GATHER))
    assert rel_err(got, oracle.apply_filter_direct(x, taps), np.abs(x).max()) <= 1e-13


@pytest.mark.parametrize("direction", ["both", "future"])
def test_non_finite_samples_at_block_boundaries(gpu_engine, direction):
    taps = oracle.tap_offsets(2000 / 130, 0.3, 2000, 0, direction)
    rng = np.random.default_rng(9)
    x = rng.standard_normal((3, 30_000))
    x[0, 9_999] = np.nan       # just before a boundary
    x[1, 10_000] = np.inf      # at it
    x[2, 10_001] = -np.inf     # just after it
    x[0, 20_000] = np.nan      # first sample of a one-sample block
    got = run_stream(gpu_engine, taps, x, [10_000, 10_000, 1, 9_999], graphs=False)
    want = gpu_engine.filter_host(x, taps, strategy=GATHER)
    assert np.isfinite(got).all()
    assert np.array_equal(got, want)
    assert (got[:, 9_999:10_002] == 0).any()


def test_storage_types_and_precision(gpu_engine):
    taps = oracle.tap_offsets(30000 / 130 * (1 + 3e-6), 4.6, 2311, 0, "future")
    rng = np.random.default_rng(2)
    base = rng.standard_normal((5, 40_000)) * 300
    sizes = block_sizes(3, base.shape[1], span_of(taps), 4096)
    for dtype in (np.int16, np.int32, np.float32):
        x = base.astype(dtype)
        got = run_stream(gpu_engine, taps, x, sizes, max_chunk=4096, graphs=False)
        assert np.array_equal(got, gpu_engine.filter_host(x, taps, strategy=GATHER)), dtype
    fp32 = run_stream(gpu_engine, taps, base, sizes, precision="fp32", max_chunk=4096,
                      graphs=False)
    assert np.array_equal(fp32, gpu_engine.filter_host(base, taps, precision="fp32",
                                                       strategy=GATHER))
    assert rel_err(fp32, oracle.apply_filter_direct(base, taps), np.abs(base).max()) <= 1e-4


def test_float32_results_and_device_tensors(gpu_engine, monkeypatch):
    import torch

    taps = oracle.tap_offsets(2000 / 130, 0.3, 2000, 0, "past")
    x = make_recording(4, 50_000, 2000, 130, seed=5)
    sizes = block_sizes(4, x.shape[1], span_of(taps), 8192)
    got32 = run_stream(gpu_engine, taps, x, sizes, max_chunk=8192, out_dtype=np.float32,
                       graphs=False)
    assert got32.dtype == np.float32
    assert np.array_equal(got32, gpu_engine.filter_host(x, taps, strategy=GATHER,
                                                        out_dtype=np.float32))
    # CUDA blocks (row views of one device tensor: row stride != block length) stay on the GPU
    d_x = torch.from_numpy(x).cuda()
    for name in ("parrm_copy_h2d_async", "parrm_copy_d2h_async", "parrm_host_copy"):
        monkeypatch.setattr(_native.lib, name, lambda *a, _n=name: pytest.fail(f"{_n} called"))
    d_got = run_stream(gpu_engine, taps, d_x, sizes, max_chunk=8192)
    monkeypatch.undo()
    assert d_got.is_cuda and d_got.dtype == torch.float64
    assert np.array_equal(d_got.cpu().numpy(), gpu_engine.filter_host(x, taps, strategy=GATHER))
    d_i16 = torch.from_numpy((x * 100).astype(np.int16)).cuda()
    got_i16 = run_stream(gpu_engine, taps, d_i16, sizes, max_chunk=8192)
    assert np.array_equal(got_i16.cpu().numpy(), gpu_engine.filter_host(
        (x * 100).astype(np.int16), taps, strategy=GATHER))


def test_two_interleaved_streams_keep_their_own_state(gpu_engine):
    a = make_recording(3, 30_000, 2000, 130, seed=1)
    b = make_recording(5, 30_000, 2000, 130, seed=2) * 7
    taps_a = oracle.tap_offsets(2000 / 130, 0.3, 2000, 0, "both")
    taps_b = oracle.tap_offsets(2000 / 130, 0.3, 1500, 0, "future")
    sa, sb = FilterStream(gpu_engine, taps_a), FilterStream(gpu_engine, taps_b)
    oa, ob = [], []
    for t in range(0, 30_000, 2_500):
        oa.append(sa.push(a[:, t:t + 2_500]))
        ob.append(sb.push(b[:, t:t + 2_500]))
    oa.append(sa.close())
    ob.append(sb.close())
    assert np.array_equal(np.concatenate(oa, 1), gpu_engine.filter_host(a, taps_a, strategy=GATHER))
    assert np.array_equal(np.concatenate(ob, 1), gpu_engine.filter_host(b, taps_b, strategy=GATHER))


@pytest.mark.parametrize("direction", ["both", "future"])
def test_graph_replay_is_bit_equal_and_eager_push_is_one_launch(gpu_engine, direction):
    taps = oracle.tap_offsets(30000 / 130 * (1 + 3e-6), 4.6, 2311, 0, direction)
    x = (make_recording(16, 60_000, 30000, 130, seed=3) * 50).astype(np.int16)
    sizes = [300] * 200
    eager = FilterStream(gpu_engine, taps, out_dtype=np.float32, graphs=False)
    graph = FilterStream(gpu_engine, taps, out_dtype=np.float32, graphs=True)
    replays0 = gpu_engine.graph_kernels
    for i, n in enumerate(sizes):
        block = x[:, i * n:(i + 1) * n]
        before = gpu_engine.launches
        e = eager.push(block)
        assert gpu_engine.launches - before == 1
        assert np.array_equal(graph.push(block), e)
    assert gpu_engine.graph_kernels - replays0 >= len(sizes) - 3 - eager.latency // 300
    assert np.array_equal(graph.close(), eager.close())


def test_public_api(gpu_engine):
    data = make_recording(6, 60_000, 2000, 130, seed=2)
    parrm = PARRM(data, 2000, 130, verbose=False)
    parrm._period = np.float64(2000 / 130 * (1 + 3e-6))
    parrm.create_filter(filter_half_width=2000, filter_direction="future")
    stream = parrm.filter_stream()
    assert stream.latency == 0
    parrm.create_filter(filter_half_width=1000, filter_direction="both")  # not seen by the stream
    outs = [stream.push(data[:, t:t + 2000]) for t in range(0, 60_000, 2000)]
    assert all(o.shape == (6, 2000) for o in outs)                 # latency 0: all final at once
    assert stream.close().shape == (6, 0)
    parrm.create_filter(filter_half_width=2000, filter_direction="future")
    assert np.array_equal(np.concatenate(outs, 1),
                          gpu_engine.filter_host(data, parrm._tap_offsets(), strategy=GATHER))

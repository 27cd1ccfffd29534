"""The float32 mode's own kernels against float64 references.

``precision="fp32"`` is not the float64 path at lower precision.  Its comb filter is compiled
for float32: other chunks ``U``, other unrolled blocks ``B``, three CTAs per SM, sometimes
another plan (``comb_e_shape``).  The gather kernels run in float32.  The search stores its
tiles in float32 and fits them in float64.  So each of these is tested here on its own terms:

* Filter: the reference is the float64 oracle on ``x.astype(float32)`` (widened exactly), the
  recording the kernel actually sees.  Only the kernel's float32 arithmetic is left in the
  difference, and every tolerance is an error model of that arithmetic (``comb_bound``,
  ``gather_bound``).  Each model must stay under 1e-4 of the input scale and under
  ``scale / (10 n_in)`` per output, so a dropped, duplicated or shifted tap, or a wrong ``n_in``
  at an edge, fails.  Every filter test forces its kernel and asserts which one ran.
* Search: the fit is float64, so the objective on a float32 tile is held to the fp64 contract
  (1e-9) against the oracle run on the tile's own values.
"""

import math

import numpy as np
import pytest

from oracle import parrm_oracle as oracle
from pyparrm_b200 import _native
from pyparrm_b200.synthetic import make_recording
from tests.test_gpu_filter import SPECIALISED_CASES, _case_taps
from tests.test_gpu_search import compare_objective

pytestmark = pytest.mark.gpu
U32 = float(np.finfo(np.float32).eps) / 2   # unit roundoff of float32 (round to nearest)
SAFETY = 1.01  # second-order terms of the models: (1 + u)^k - 1 - k u, k <= 5 000 -> < 1e-4 k u
COMB, GATHER_SMEM, GATHER_GLOBAL = ("parrm_filter_comb_e", "filter_gather_smem_kernel",
                                    "filter_gather_global_kernel")


class CombShape:
    """The float32 specialisation of a tap set, as ``parrm_filter_specialise_check`` reports
    it (no GPU, nothing compiled), plus every offset the kernel loads, with multiplicity."""

    def __init__(self, taps):
        plan, desc = _native.plan_filter(taps, _native.F32)
        assert desc["kind"] == 1
        shape = np.zeros(12, dtype=np.int32)
        _native.check(_native.lib.parrm_filter_specialise_check(
            plan.ctypes.data, _native.F32, None, shape.ctypes.data, None),
            "parrm_filter_specialise_check")
        self.d, self.nk, self.m0, self.m1, self.nb0, self.nb1, self.n_single, self.u = (
            int(v) for v in shape[:8])
        self.ctas = int(shape[9])
        self.b = self.u * -(-self.m0 // self.u)   # unrolled block: steps between re-adds
        self.n_taps = len(taps)
        loads = [a + q * desc["stride"] for m, boxes in zip(desc["windows"], desc["boxes"])
                 for a in boxes for q in range(m)]
        loads += list(desc["plus"]) + list(desc["minus"]) + [0] * abs(desc["centre"])
        self.loads = np.asarray(loads, dtype=np.int64)
        # deepest chain of roundings any load goes through when the sums are re-added: half
        # its pattern sum (two partial chains), the ring sum of M_k values, S0 + S1, + singles
        depth1 = math.ceil(self.nb1 / 2) + self.m1 if self.nk > 1 else 0
        self.depth = max(math.ceil(self.nb0 / 2) + self.m0, depth1, self.n_single + 1) + 2

    def __str__(self):
        return (f"d {self.d}, M {self.m0}/{self.m1}, U {self.u}, B {self.b}, "
                f"{self.ctas} CTAs/SM, {self.n_taps} taps, {len(self.loads)} loads")


def comb_bound(x, taps, cs, scale):
    """Worst-case error of each output of the float32 comb kernel, ``[T]``.

    ``tot`` is a sum of the loads in range: ``L`` of them, each ``|x| <= scale``.  A sum over a
    tree of additions errs by at most ``u`` times the sum, over its leaves, of ``|leaf|`` times
    the leaf's depth, so re-adding ``tot`` from the rings costs ``depth * L * u * scale``.
    Between re-adds a running sum takes two more updates per step, each rounded to ``u`` times
    the window sum (``<= L scale``), for at most one block of ``B`` steps: ``+ 2B L u scale``.
    That holds for outputs whose whole tap window is in range (``n_in = n_taps``).  At the
    recording edges the float32 kernel re-adds on every step (the window empties there while
    the running sum would still carry the full window's rounding), so no drift term.  The
    output ``x - tot / n_in`` adds the rounding of ``1/n_in``, of the product and of the result:
    ``(2 L / n_in + |y| / scale) u scale`` with ``|y| <= scale (1 + L / n_in)``.  In all:

        err(t) <= u scale [(depth + 2B [n_in = n_taps] + 3) L(t) / n_in(t) + 1]

    with ``L(t)`` the loads in range of output ``t`` (all loads for interior outputs).
    ``depth``, ``B`` and ``L`` come from the specialisation; 0 where ``n_in = 0``.
    """
    n = x.shape[1]
    n_in = oracle.in_range_tap_count(n, taps)
    full = n_in == cs.n_taps
    loads = np.where(full, len(cs.loads), oracle.in_range_tap_count(n, cs.loads))
    with np.errstate(divide="ignore", invalid="ignore"):
        rel = (cs.depth + 2 * cs.b * full + 3) * loads / n_in + 1
    return np.where(n_in > 0, SAFETY * U32 * scale * rel, 0.0)


def gather_bound(x, taps):
    """Running error bound of the float32 gather kernels (and of the comb kernel's tap-by-tap
    re-evaluation of non-finite windows), ``[C, T]``.

    They add the in-range taps one by one in ascending order, so the sum errs by at most
    ``u * sum_k |s_k|`` over its partial sums ``s_k``; the division by ``n_in`` (exact in
    float32) and the subtraction round once each.  With the exact partial sums of the
    float32 samples:

        err(t) <= u (sum_k |s_k| / n_in + 2 |s_n| / n_in + |x[t]|)

    The a-priori form of this (``|s_k| <= k scale``: ``(n_in + 1) / 2 * u scale``) would pass a
    dropped tap for more than ~1 800 taps, the huge-span case here has 3 000; the partial sums
    of the actual recording keep the bound far below that on zero-mean data.
    """
    n = x.shape[1]
    acc = np.zeros_like(x)
    path = np.zeros_like(x)
    with np.errstate(invalid="ignore", over="ignore"):
        for w in taps.astype(np.int64):
            lo, hi = max(0, w), min(n, n + w)
            if lo < hi:
                acc[:, lo:hi] += x[:, lo - w: hi - w]
                path[:, lo:hi] += np.abs(acc[:, lo:hi])
        n_in = oracle.in_range_tap_count(n, taps)
        bound = SAFETY * U32 * ((path + 2 * np.abs(acc)) / np.maximum(n_in, 1) + np.abs(x))
    return np.where(n_in > 0, bound, 0.0)


def check_limits(bound, taps, scale, label):
    """A bound is only worth its name if it resolves one tap and meets the 1e-4 contract."""
    n_in = oracle.in_range_tap_count(bound.shape[-1], taps)
    ok = n_in > 0
    rel = np.nan_to_num(bound / scale, nan=np.inf).reshape(-1, bound.shape[-1])
    assert rel.max() <= 1e-4, f"{label}: bound {rel.max():.2e} exceeds the 1e-4 contract"
    worst = (rel[:, ok] * 10 * n_in[ok]).max() if ok.any() else 0.0
    assert worst < 1.0, f"{label}: bound would pass a dropped tap ({worst:.2f} of scale / 10 n_in)"
    return float(rel.max())


def rounded(x):
    """The recording as the float32 kernels see it, widened back exactly."""
    with np.errstate(over="ignore"):
        return x.astype(np.float32).astype(np.float64)


def finite_scale(x):
    finite = np.abs(x[np.isfinite(x)])
    return max(float(finite.max()) if finite.size else 0.0, 1e-30)


def check_filtered(got, x64, taps, bound, label, scale):
    """``got`` against the oracle on the rounded recording ``x64``, output by output."""
    want = oracle.apply_filter_direct(x64, taps)
    err = np.abs(got - want)
    assert np.all(err <= bound), (
        f"{label}: error {err.max() / scale:.2e} of the scale at "
        f"{np.unravel_index(np.argmax(err - bound), err.shape)}, bound there "
        f"{bound.flat[np.argmax(err - bound)] / scale:.2e}")
    return float(err.max() / scale) if err.size else 0.0


def run_device(engine, x32, taps, kernel):
    import torch

    got = engine.filter_device(torch.from_numpy(x32).cuda(), taps, kernel=kernel)
    assert got.dtype == torch.float32
    return got.double().cpu().numpy()


# ---------------------------------------------------------------------------------------------
# 1. the specialised float32 kernel, every case, every shape
SHAPES = [(3, 50_000), (1, 7001), (2, 1999), (5, 20_011), (160, 30_000)]


@pytest.mark.parametrize("name", list(SPECIALISED_CASES))
def test_specialised_fp32_every_case_and_shape(gpu_engine, name):
    """The shapes of the float64 test (interior blocks, edges, recordings shorter than the tap
    window, one strip and many) plus one long row of int16-like counts with a DC offset, where
    the running sums are large and meet many blocks."""
    taps = _case_taps(name)
    cs = CombShape(taps)
    rng = np.random.default_rng(len(name) + 32)
    inputs = [rng.standard_normal(shape) * 3 + 10 for shape in SHAPES]
    inputs.append(np.round(rng.standard_normal((1, 1_200_003)) * 300 + 2000))
    for x in inputs:
        x32 = x.astype(np.float32)
        x64 = x32.astype(np.float64)
        got = run_device(gpu_engine, x32, taps, _native.KERNEL_SPECIALISED)
        assert gpu_engine.last_filter_kernel == COMB
        scale = finite_scale(x64)
        bound = comb_bound(x64, taps, cs, scale)
        limit = check_limits(bound, taps, scale, name)
        worst = check_filtered(got, x64, taps, bound, f"{name} {x.shape}", scale)
        print(f"fp32 comb {name} [{cs}] {x.shape}: worst {worst:.2e}, bound {limit:.2e} "
              "of the input scale")


# ---------------------------------------------------------------------------------------------
# 2. rows that start off 16-byte alignment (the chunk grid is in units of 4 elements)
@pytest.mark.parametrize("name", ["cfg2", "cfg4 future", "short future"])
def test_specialised_fp32_unaligned_rows(gpu_engine, name):
    import torch

    taps = _case_taps(name)
    cs = CombShape(taps)
    rng = np.random.default_rng(7)
    n, ld = 30_001, 30_006   # ld % 4 == 2: neighbouring rows start at other alignments too
    x32 = (rng.standard_normal((4, n)) * 3 + 10).astype(np.float32)
    x64 = x32.astype(np.float64)
    scale = finite_scale(x64)
    bound = comb_bound(x64, taps, cs, scale)
    check_limits(bound, taps, scale, name)
    for offset in (1, 2, 3):
        buf = torch.zeros(4 * ld + offset, dtype=torch.float32, device="cuda")
        d_x = buf[offset:].as_strided((4, n), (ld, 1))
        d_x.copy_(torch.from_numpy(x32))
        assert d_x.data_ptr() % 16 == 4 * offset
        got = gpu_engine.filter_device(d_x, taps, kernel=_native.KERNEL_SPECIALISED)
        assert gpu_engine.last_filter_kernel == COMB
        worst = check_filtered(got.double().cpu().numpy(), x64, taps, bound,
                               f"{name} offset {offset}", scale)
        print(f"fp32 comb {name} rows at element offset {offset}: worst {worst:.2e}")


# ---------------------------------------------------------------------------------------------
# 3. time windows (x_t0 / t0 / n_out), as sharding cuts a channel in time
@pytest.mark.parametrize("name", ["cfg2", "cfg4 future"])
def test_specialised_fp32_time_shards_stitch(gpu_engine, monkeypatch, name):
    from pyparrm_b200 import _sharding

    taps = _case_taps(name)
    cs = CombShape(taps)
    x = make_recording(1, 200_003, 2000, 130, seed=3)
    x64 = rounded(x)
    scale = finite_scale(x64)
    bound = comb_bound(x64, taps, cs, scale)
    check_limits(bound, taps, scale, name)
    w_lo, w_hi = min(int(taps[0]), 0), max(int(taps[-1]), 0)
    monkeypatch.setenv("PYPARRM_B200_FILTER_KERNEL", str(_native.KERNEL_SPECIALISED))
    for world in (3, 4):
        got = np.full_like(x, np.nan)
        for c0, c1, t0, t1, x0, x1 in _sharding.channel_or_time_shards(1, x.shape[1], world,
                                                                        w_lo, w_hi):
            shard = gpu_engine.filter_shard(x[c0:c1, x0:x1], taps, x0, t0, t1, x.shape[1],
                                            precision="fp32")
            assert gpu_engine.last_filter_kernel == COMB
            got[c0:c1, t0:t1] = shard.cpu().numpy()
        worst = check_filtered(got, x64, taps, bound, f"{name}, {world} shards", scale)
        print(f"fp32 comb {name}, {world} time shards: worst {worst:.2e}")


# ---------------------------------------------------------------------------------------------
# 4. non-finite samples and outliers, both kernels
@pytest.mark.parametrize("name", ["cfg2", "cfg4 past"])
def test_fp32_non_finite_samples_and_outliers(gpu_engine, name):
    """NaN, +Inf, -Inf and a float64 value above FLT_MAX (Inf once converted) zero exactly the
    outputs the reference finds non-finite on the converted recording; every other output
    meets its bound.  A 1e12 outlier leaves ~1e12 eps32 of rounding in the comb kernel's
    running sums until the next re-add: outputs more than one block (``B d`` samples) past
    its window must meet the bound of the rest of the row; inside that block the error is
    held to the same model with the outlier as the scale, and printed (DESIGN 4.1)."""
    taps = _case_taps(name)
    cs = CombShape(taps)
    rng = np.random.default_rng(9)
    x = rng.standard_normal((4, 60_000))
    x[0, 12_345] = np.nan
    x[1, 30_000] = np.inf
    x[1, 30_007] = -np.inf
    x[2, 40_000] = 1e39           # above FLT_MAX: +Inf in float32
    p = 20_000
    x[3, p] = 1e12
    x64 = rounded(x)
    x32 = x64.astype(np.float32)
    assert np.isinf(x32[2, 40_000])
    with np.errstate(invalid="ignore"):
        want = oracle.apply_filter_direct(x64, taps)
    bad = ~np.isfinite(want)
    assert bad[:3].any(axis=1).all()
    want[bad] = 0.0
    rest = np.ones(x.shape[1], dtype=bool)
    rest[p] = False
    scale = finite_scale(x64[:, rest])                     # everything but the outlier
    b_gather = gather_bound(x64, taps)
    b_comb = np.maximum(comb_bound(x64, taps, cs, scale), b_gather)  # flagged spans: tap by tap
    check_limits(comb_bound(x64, taps, cs, scale), taps, scale, name)
    # outputs whose running sums may hold the outlier: from its first load to one block past
    # its last one
    lo, hi = p + int(cs.loads.min()), p + int(cs.loads.max())
    after = np.zeros(x.shape[1], dtype=bool)
    after[max(lo, 0): hi + cs.b * cs.d + 1] = True
    inside = np.zeros(x.shape[1], dtype=bool)
    inside[np.unique(p + np.concatenate([taps, [0]]))] = True
    for kernel, kname in ((_native.KERNEL_SPECIALISED, COMB), (_native.KERNEL_GATHER, GATHER_SMEM)):
        got = run_device(gpu_engine, x32, taps, kernel)
        assert gpu_engine.last_filter_kernel == kname
        assert np.isfinite(got).all()
        assert np.all(got[bad] == 0), kname
        err = np.abs(got - want)
        bound = b_comb if kernel == _native.KERNEL_SPECIALISED else b_gather
        assert np.all(err[:3][~bad[:3]] <= bound[:3][~bad[:3]]), (kname, (err[:3] - bound[:3]).max())
        # the outlier row: every output of the gather meets its running bound; the comb kernel
        # past the outlier's reach meets the bound of the rest of the row
        if kernel == _native.KERNEL_GATHER:
            assert np.all(err[3] <= b_gather[3]), kname
        else:
            assert np.all(err[3, ~after] <= bound[3, ~after]), kname
            # within its reach: the same model, with the outlier as the scale
            assert np.all(err[3, after] <= comb_bound(x64[3:], taps, cs, 1e12)[after]), kname
        residue = after & ~inside
        print(f"fp32 {kname} {name}: worst {err[:3][~bad[:3]].max() / scale:.2e} of the input scale; "
              f"1e12 outlier: {err[3, inside].max():.3g} inside its window, "
              f"{err[3, residue].max():.3g} in the block after it "
              f"({err[3, residue].max() / scale:.2e} of the rest of the row, "
              f"{err[3, residue].max() / 1e12:.2e} of the outlier), "
              f"{err[3, ~after].max() / scale:.2e} elsewhere")


# ---------------------------------------------------------------------------------------------
# 5. the gather kernels in float32
@pytest.mark.parametrize("shape", [(1, 1), (1, 2), (3, 17), (2, 1023), (5, 4096), (1, 4097),
                                   (2, 12289), (7, 20001), (0, 10), (2, 0)])
def test_gather_fp32_shared_memory(gpu_engine, shape):
    rng = np.random.default_rng(shape[0] * 131 + shape[1])
    x32 = (rng.standard_normal(shape) * 3 + 100.0).astype(np.float32)
    x64 = x32.astype(np.float64)
    per = 15.3846
    for direction, hw, omit in (("both", 2000, 0), ("past", 777, 3), ("future", 50, 0)):
        taps = oracle.tap_offsets(per, per / 50, hw, omit, direction)
        if not x32.size:   # nothing to launch; the host entry point returns the empty shape
            assert gpu_engine.filter_host(x32, taps, precision="fp32").shape == shape
            continue
        got = run_device(gpu_engine, x32, taps, _native.KERNEL_GATHER)
        assert got.shape == shape
        assert gpu_engine.last_filter_kernel == GATHER_SMEM
        scale = finite_scale(x64)
        bound = gather_bound(x64, taps)
        check_limits(bound, taps, scale, f"{shape} {direction}")
        check_filtered(got, x64, taps, bound, f"{shape} {direction}", scale)


def test_gather_fp32_global_memory_huge_span(gpu_engine):
    rng = np.random.default_rng(1)
    x32 = rng.standard_normal((2, 90_000)).astype(np.float32)
    x64 = x32.astype(np.float64)
    taps = oracle.tap_offsets(230.77, 4.6, 40_000, 0, "both")
    got = run_device(gpu_engine, x32, taps, _native.KERNEL_GATHER)
    assert gpu_engine.last_filter_kernel == GATHER_GLOBAL
    scale = finite_scale(x64)
    bound = gather_bound(x64, taps)
    limit = check_limits(bound, taps, scale, "huge span")
    worst = check_filtered(got, x64, taps, bound, "huge span", scale)
    print(f"fp32 global gather, {len(taps)} taps: worst {worst:.2e}, bound {limit:.2e}")


# ---------------------------------------------------------------------------------------------
# 6. the host pipeline in float32 through a ring of many chunks
def _storage(kind, base):
    if kind == "float64":
        return base
    if kind == "float32":
        return base.astype(np.float32)
    if kind == "int16":
        return np.round(base).astype(np.int16)
    return (np.round(base) + 30_000_000).astype(np.int32)  # above 2^24: rounds on widening


@pytest.mark.parametrize("kind", ["float64", "float32", "int16", "int32"])
def test_host_pipeline_fp32_multi_chunk(gpu_engine, monkeypatch, kind):
    """1.5 MB chunks: 6 x 300 000 goes in one channel per chunk (the three slots are reused),
    one 2 M-sample row in time chunks with halos.  Both kernels, float64 and float32 out."""
    from pyparrm_b200 import _engine

    monkeypatch.setattr(_engine, "_CHUNK_BYTES", 3 << 19)
    taps = _case_taps("cfg2")
    cs = CombShape(taps)
    rng = np.random.default_rng(6)
    for shape in ((6, 300_000), (1, 2_000_000)):
        x = _storage(kind, rng.standard_normal(shape) * 300)
        x64 = rounded(x.astype(np.float64))   # widened to float32 on the device
        scale = finite_scale(x64)
        bounds = {COMB: comb_bound(x64, taps, cs, scale), GATHER_SMEM: gather_bound(x64, taps)}
        for kernel, kname in ((_native.KERNEL_SPECIALISED, COMB), (_native.KERNEL_GATHER, GATHER_SMEM)):
            check_limits(bounds[kname], taps, scale, f"{kind} {kname}")
            monkeypatch.setenv("PYPARRM_B200_FILTER_KERNEL", str(kernel))
            per_chunk = 1 + (kind != "float32") + 1   # widen in, the kernel, widen out
            launches = gpu_engine.launches
            out = gpu_engine.filter_host(x, taps, precision="fp32")
            chunks = (gpu_engine.launches - launches) / per_chunk
            assert gpu_engine.last_filter_kernel == kname
            assert out.dtype == np.float64 and chunks >= 4, (kind, shape, chunks)
            worst = check_filtered(out, x64, taps, bounds[kname], f"{kind} {shape} {kname}", scale)
            # float32 out: same arithmetic, but time chunks twice as long where the output was
            # the widest element, so the comb strips may start at other samples
            out32 = gpu_engine.filter_host(x, taps, precision="fp32", out_dtype=np.float32)
            assert out32.dtype == np.float32 and gpu_engine.last_filter_kernel == kname
            worst32 = check_filtered(out32.astype(np.float64), x64, taps, bounds[kname],
                                     f"{kind} {shape} {kname} float32 out", scale)
            print(f"fp32 host pipeline {kind} {shape} {kname}: {chunks:.0f} chunks, worst "
                  f"{worst:.2e} (float32 out {worst32:.2e})")


# ---------------------------------------------------------------------------------------------
# 7. the search on float32 tiles: stored in float32, fitted in float64
def _fit_input(data, tile, idx):
    """Standardised recording whose fitted columns are the float32 tile's own values."""
    z = oracle.standardise(data, 3.0)
    z[:, idx] = tile.y.double().cpu().numpy().T
    return z


def test_fp32_tiles_are_the_rounded_fp64_tiles(gpu_engine):
    import torch

    for n_chans in (1, 2, 65):
        data = make_recording(n_chans, 70_001, 2000, 130, seed=21 + n_chans)
        idx_sets = [np.arange(100, 5101),
                    np.unique(np.random.default_rng(0).integers(0, 69_000, 20_000)) + 500]
        t64 = gpu_engine.prepare_tiles(data, idx_sets, 3.0)
        t32 = gpu_engine.prepare_tiles(data, idx_sets, 3.0, precision="fp32")
        for a, b in zip(t64, t32):
            assert b.y.dtype == torch.float32 and b.y.shape == a.y.shape
            assert torch.equal(b.y, a.y.to(torch.float32))
            y = b.y.double().cpu().numpy()
            want = (y ** 2).sum(axis=0)
            assert np.abs(b.sumsq.cpu().numpy() - want).max() <= 1e-13 * want.max()


def test_fp32_evaluator_channel_counts(gpu_engine):
    """Narrow kernel (1, 2 channels), tensor kernel, one full channel tile (64), re-tiled
    layouts (3, 65, 130)."""
    base = make_recording(130, 12_000, 2000, 130, seed=13)
    idx = np.arange(1000, 6001)
    periods = 2000 / 130 * (1 + np.array([-2e-3, 0.0, 3e-6, 1e-3]))
    for n_chans in (1, 2, 3, 64, 65, 130):
        data = np.ascontiguousarray(base[:n_chans])
        (tile,) = gpu_engine.prepare_tiles(data, [idx], 3.0, precision="fp32")
        got = gpu_engine.evaluate(tile, periods, 10, 1.0, n_chans)
        want = oracle.objective_many(periods, _fit_input(data, tile, idx), idx, 10, 1.0, n_chans,
                                     n_jobs=8)
        worst = compare_objective(got, want, f"fp32 tile, {n_chans} channels", periods, idx, 10)
        print(f"fp32 tile, {n_chans} channels: worst relative error {worst:.2e}")


@pytest.mark.parametrize("bandwidth", [1, 4, 7, 12, 16, 23])
def test_fp32_evaluator_row_blocks(gpu_engine, bandwidth):
    base = make_recording(6, 9_000, 2000, 130, seed=17)
    idx = np.arange(700, 700 + 128 * 9 + 37)
    periods = 2000 / 130 * (1 + np.array([-1.5e-3, 2e-6, 7e-4]))
    for n_chans in (1, 3, 6):
        data = np.ascontiguousarray(base[:n_chans])
        (tile,) = gpu_engine.prepare_tiles(data, [idx], 3.0, precision="fp32")
        got = gpu_engine.evaluate(tile, periods, bandwidth, 1.0, n_chans)
        want = oracle.objective_many(periods, _fit_input(data, tile, idx), idx, bandwidth, 1.0,
                                     n_chans, n_jobs=4)
        compare_objective(got, want, f"fp32 bw {bandwidth}, {n_chans} ch", periods, idx, bandwidth)


def test_fp32_evaluator_few_and_many_candidates(gpu_engine):
    """Few candidates split the samples over CTAs; many get one CTA each."""
    data = make_recording(3, 60_000, 2000, 130, seed=12)
    idx = np.arange(10_000, 35_001)
    (tile,) = gpu_engine.prepare_tiles(data, [idx], 3.0, precision="fp32")
    z = _fit_input(data, tile, idx)
    periods = 2000 / 130 * (1 + np.linspace(-1e-3, 1e-3, 700))
    many = gpu_engine.evaluate(tile, periods, 20, 1.0, 3)
    pick = np.arange(0, 700, 35)
    want = oracle.objective_many(periods[pick], z, idx, 20, 1.0, 3, n_jobs=8)
    compare_objective(many[pick], want, "fp32 tile, 700 candidates", periods[pick], idx, 20)
    for few in (periods[:1], periods[[0, 350, 699]]):
        got = gpu_engine.evaluate(tile, few, 20, 1.0, 3)
        want = oracle.objective_many(few, z, idx, 20, 1.0, 3, n_jobs=4)
        compare_objective(got, want, f"fp32 tile, {len(few)} candidates", few, idx, 20)


def test_fp32_evaluator_large_sample_indices(gpu_engine):
    n_chans, n = 2, 1_200_000
    data = make_recording(n_chans, n, 2000, 130, seed=21)
    rng = np.random.default_rng(3)
    per = 2000 / 130 * (1 + 3e-6)
    periods = per * (1 + np.array([-2e-3, -1e-5, 0.0, 3e-6, 4e-4]))
    for idx in (np.arange(1_100_000, 1_105_001),
                np.unique(rng.integers(0, n - 60_002, 6000)) + 30_000):
        (tile,) = gpu_engine.prepare_tiles(data, [idx], 3.0, precision="fp32")
        got = gpu_engine.evaluate(tile, periods, 20, 1.0, n_chans)
        want = oracle.objective_many(periods, _fit_input(data, tile, idx), idx, 20, 1.0, n_chans,
                                     n_jobs=4)
        compare_objective(got, want, "fp32 tile, large indices", periods, idx, 20)


def test_fp32_device_nelder_mead_retraces_host_state_machines(gpu_engine):
    """csrc/neldermead.cu on float32 tiles vs pyparrm_b200/_neldermead.py driven by the same
    evaluator with the same batch shape: every chain bit-equal."""
    from pyparrm_b200._neldermead import fmin_batch

    data = make_recording(3, 40_000, 2000, 130, seed=12)
    for idx, bw, lam, starts in (
        (np.arange(5_000, 10_001), 5, 1.0, [15.38, 15.3846, 15.40, 15.2, 15.39]),
        (np.arange(100, 1_100), 10, 1.0, [7.7, 15.5]),
    ):
        (tile,) = gpu_engine.prepare_tiles(data, [idx], 3.0, precision="fp32")
        assert tile.y_code == _native.F32
        n = len(starts)

        def evaluate(p, tile=tile, n=n, bw=bw, lam=lam):
            padded = np.resize(np.asarray(p, dtype=np.float64), 5 * n)  # same launch shape
            return gpu_engine.evaluate(tile, padded, bw, lam, 3)[: len(p)]

        want = fmin_batch(evaluate, starts)
        got = gpu_engine.nm_minimise(tile, starts, bw, lam, 3)
        for g, w in zip(got, want):
            assert g[0] == w[0] and (g[1] == w[1] or (np.isnan(g[1]) and np.isnan(w[1])))
            assert g[2:] == (w[2], w[3]), (g, w)

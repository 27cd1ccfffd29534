"""Filter planner (host side of the C ABI) and the specialised kernel's design, on the CPU.

The planner regroups the tap set of ``_generate_filter`` (parrm.py:803-833) into comb boxes
plus single taps (pyparrm_b200/csrc/filter_plan.h).  That is only legal if it is an identity
over integers, so every plan is expanded back and compared with the tap set, bit for bit.
"""

import ctypes

import numpy as np
import pytest

from oracle import parrm_oracle as oracle
from pyparrm_b200 import _native
from tests.pattern_model import PatternModel


def expand(desc, lo, hi):
    acc = np.zeros(hi - lo + 1, dtype=np.int64)
    for m, boxes in zip(desc["windows"], desc["boxes"]):
        for a in boxes:
            for q in range(m):
                acc[a + q * desc["stride"] - lo] += 1
    for w in desc["plus"]:
        acc[w - lo] += 1
    for w in desc["minus"]:
        acc[w - lo] -= 1
    acc[0 - lo] += desc["centre"]
    return acc


CASES = [
    # period, phw, hw, omit, direction   (BASELINE configs first)
    (2000 / 130 * (1 + 3e-6), None, 2000, 0, "both"),
    (1000 / 145 * (1 + 3e-6), None, 2469, 0, "both"),
    (30000 / 130 * (1 + 3e-6), None, 2311, 0, "past"),
    (30000 / 130 * (1 + 3e-6), None, 2311, 0, "future"),
    (1.3311148014466094, 0.01, 2000, 20, "both"),
    (1.3311148014466094, None, 2000, 0, "both"),
    (15.3846, None, 777, 3, "past"),
    (15.3846, None, 50, 0, "future"),
    (2.0, None, 40, 0, "both"),
    (7.123456, 0.9, 3000, 100, "both"),
    (101.5, 3.3, 5000, 0, "both"),
    (230.77, 4.6, 40_000, 0, "both"),
    (2000 / 130 * (1 + 3e-6), None, 1500, 300, "both"),
]


@pytest.mark.parametrize("case", CASES)
def test_plans_are_exact_regroupings(case):
    period, phw, hw, omit, direction = case
    taps = oracle.tap_offsets(period, period / 50 if phw is None else phw, hw, omit, direction)
    for strategy in (_native.PLAN_AUTO, _native.PLAN_GATHER):
        _, desc = _native.plan_filter(taps, strategy=strategy)
        assert desc["n_taps"] == len(taps)
        if strategy == _native.PLAN_GATHER:
            assert desc["kind"] == 0
        if desc["kind"] == 0:
            continue
        lo, hi = min(int(taps[0]), 0), max(int(taps[-1]), 0)
        want = np.zeros(hi - lo + 1, dtype=np.int64)
        want[taps - lo] = 1
        assert np.array_equal(expand(desc, lo, hi), want)
        n_terms = sum(len(b) for b in desc["boxes"]) + len(desc["plus"]) + len(desc["minus"])
        assert n_terms <= 120 and desc["cost"] < 0.6 * len(taps)
        assert desc["centre"] <= 0 and len(desc["windows"]) in (1, 2)


def test_baseline_configs_get_short_plans():
    """cfg2 (160 taps) must cost ~10 loads, not 160: that is what the roofline target needs."""
    period = 2000 / 130 * (1 + 3e-6)
    taps = oracle.tap_offsets(period, period / 50, 2000, 0, "both")
    _, desc = _native.plan_filter(taps)
    assert desc["kind"] == 1 and desc["stride"] == 200 and sorted(desc["windows"]) == [10, 20]
    assert sum(len(b) for b in desc["boxes"]) + len(desc["plus"]) + len(desc["minus"]) <= 12
    # the other named tap sets: cfg3 198 taps, cfg4 95 one-sided taps
    for fs, fa, hw, direction, most in ((1000, 145, 2469, "both", 10), (30000, 130, 2311, "past", 16)):
        period = fs / fa * (1 + 3e-6)
        _, desc = _native.plan_filter(oracle.tap_offsets(period, period / 50, hw, 0, direction))
        n_terms = sum(len(b) for b in desc["boxes"]) + len(desc["plus"]) + len(desc["minus"])
        assert desc["kind"] == 1 and 64 <= desc["stride"] <= 992 and n_terms <= most


RUNNABLE_CASES = CASES + [
    (1.3311148014466094, None, 2408, 0, "both"),  # the bundled example, create_filter() defaults
    (8.6613, None, 5000, 0, "both"),              # long windows on a stride of 537
    (2000 / 130, 1.0, 2000, 0, "both"),           # runs of consecutive taps
    (30000 / 130, 20.0, 5000, 0, "past"),
    (7.3, 0.5, 300, 5, "future"),
]


@pytest.mark.parametrize("case", RUNNABLE_CASES)
def test_comb_plans_are_runnable(case):
    """Whatever comb plan the planner returns, the specialised kernel must accept: the planner
    bounds the box lengths by the registers the kernel has at that stride (a stride of 800 is an
    832-thread CTA: 72 registers per thread, rings of at most ten float64 values), instead of
    returning the cheapest plan and leaving the job to the tap-by-tap gather."""
    period, phw, hw, omit, direction = case
    taps = oracle.tap_offsets(period, period / 50 if phw is None else phw, hw, omit, direction)
    new_case = case not in CASES
    for dtype in (_native.F64, _native.F32) if new_case or len(taps) < 400 else (_native.F64,):
        plan, desc = _native.plan_filter(taps, dtype)
        if desc["kind"] != 1:
            continue
        shape = np.zeros(12, dtype=np.int32)
        # range check for every case; the new float64 plans are also compiled (NVRTC, no GPU
        # needed) except the 860-tap one, whose build takes ~25 s (it is built and run in
        # tests/test_gpu_filter.py)
        compiled = ctypes.c_size_t(0)
        build = new_case and dtype == _native.F64 and len(taps) < 800
        status = _native.lib.parrm_filter_specialise_check(
            plan.ctypes.data, dtype, None, shape.ctypes.data,
            ctypes.byref(compiled) if build else None)
        assert status == 0, (case, dtype, desc["stride"], desc["windows"], _native.last_error())
        assert compiled.value > 0 or not build
        if case in CASES and dtype == _native.F64:
            continue  # expanded in test_plans_are_exact_regroupings
        lo, hi = min(int(taps[0]), 0), max(int(taps[-1]), 0)
        want = np.zeros(hi - lo + 1, dtype=np.int64)
        want[taps - lo] = 1
        assert np.array_equal(expand(desc, lo, hi), want)
    # the BASELINE tap sets and the five realistic ones added above must not end on the gather
    if case in CASES[:5] or case in RUNNABLE_CASES[len(CASES):]:
        assert _native.plan_filter(taps, _native.F64)[1]["kind"] == 1, case


def test_random_tap_sets():
    rng = np.random.default_rng(7)
    for _ in range(40):
        n = int(rng.integers(1, 300))
        taps = np.unique(rng.integers(-3000, 3000, n))
        taps = taps[taps != 0].astype(np.int32)
        if len(taps) == 0:
            continue
        _, desc = _native.plan_filter(taps)
        if desc["kind"] == 1:
            lo, hi = min(int(taps[0]), 0), max(int(taps[-1]), 0)
            want = np.zeros(hi - lo + 1, dtype=np.int64)
            want[taps - lo] = 1
            assert np.array_equal(expand(desc, lo, hi), want)
    one, blob = np.array([5], dtype=np.int32), np.zeros(4096, dtype=np.uint8)
    status = _native.lib.parrm_filter_plan(one.ctypes.data, 1, 0, _native.PLAN_COMB,
                                           blob.ctypes.data, 4096)
    assert status == 4 and "comb" in _native.last_error()


MODEL_CASES = [
    # case index, recording length, steps per chunk, gamma, pieces, time chunk
    (0, 30_011, 5, 1, 3, None),
    (0, 700, 10, 0, 1, None),
    (0, 20_000, 3, 0, 2, None),          # block longer than the box (B = 21 > M0 = 20)
    (0, 40_000, 10, 1, 2, (9_000, 21_000)),
    (1, 30_000, 7, 0, 2, None),          # cfg3: M0 = 25, B = 28
    (2, 20_000, 8, 0, 2, None),          # cfg4, documented "past"
    (3, 20_000, 8, 1, 1, None),
    (4, 19_130, 3, 0, 1, None),
    (12, 15_000, 4, 0, 3, (0, 7_000)),
]


@pytest.mark.parametrize("spec", MODEL_CASES)
def test_pattern_first_design_matches_oracle(spec):
    """Chunk grid, priming block, register rings of the unrolled block, sliding sums, piece
    boundaries and edge counts of the run-time specialised kernel (NumPy model with its index
    arithmetic, tests/pattern_model.py) against the oracle's direct sum."""
    case, n_total, u, gamma, pieces, chunk = spec
    period, phw, hw, omit, direction = CASES[case]
    taps = oracle.tap_offsets(period, period / 50 if phw is None else phw, hw, omit, direction)
    _, desc = _native.plan_filter(taps, strategy=_native.PLAN_COMB)
    rng = np.random.default_rng(case)
    x = rng.standard_normal((1, n_total)) + 3.0
    want = oracle.apply_filter_direct(x, taps)[0]
    model = PatternModel(taps, desc, u)
    if chunk is None:
        got = model.run(x[0], 0, 0, n_total, n_total, gamma, pieces)
    else:
        t0, t1 = chunk
        x0, x1 = max(0, t0 - model.w_hi), min(n_total, t1 - model.w_lo)
        got = model.run(x[0, x0:x1], x0, t0, t1 - t0, n_total, gamma, pieces)
        want = want[t0:t1]
    assert not np.isnan(got).any()
    assert np.abs(got - want).max() <= 1e-12


@pytest.mark.parametrize("case", [0, 2, 4])
def test_pattern_first_non_finite_window(case):
    """A NaN / Inf sample zeroes exactly the outputs whose tap window (or own sample) holds
    it -- parrm.py:869's isfinite -> 0 applied per output -- and outputs past the window are
    exact again (the running sums are re-added from the rings while they are non-finite)."""
    period, phw, hw, omit, direction = CASES[case]  # cfg4 and cfg1 plans carry -1 terms
    taps = oracle.tap_offsets(period, period / 50 if phw is None else phw, hw, omit, direction)
    _, desc = _native.plan_filter(taps, strategy=_native.PLAN_COMB)
    rng = np.random.default_rng(3)
    x = rng.standard_normal((1, 40_000))
    x[0, 12_345] = np.nan
    x[0, 30_000] = np.inf
    x[0, 5] = 1e12
    with np.errstate(invalid="ignore"):
        want = oracle.apply_filter_direct(x, taps)[0]
    want[~np.isfinite(want)] = 0.0
    got = PatternModel(taps, desc, 8).run(x[0], 0, 0, 40_000, 40_000, 0, 2)
    assert np.isfinite(got).all()
    assert np.array_equal(got == 0, want == 0)
    assert np.abs(got - want).max() <= 1e-3  # 1e12 outlier: rounding residue ~1e12 * 2^-52 * steps


def test_fp32_specialisations_the_gpu_tests_rely_on():
    """tests/test_gpu_fp32.py runs the float32 comb kernel on the tap sets of
    tests/test_gpu_filter.py because float32 gets specialisations that float64 does not
    (comb_e_shape picks the chunk, the block and the CTAs per SM from the element size).  This
    asserts that those cases still reach what that file claims for them, with the shape check
    alone (nothing compiled): if the shape choice changes, it names the coverage that moved."""
    from tests.test_gpu_filter import SPECIALISED_CASES, _case_taps

    def shape(name, dtype):
        plan, _ = _native.plan_filter(_case_taps(name), dtype)
        s = np.zeros(12, dtype=np.int32)
        status = _native.lib.parrm_filter_specialise_check(plan.ctypes.data, dtype, None,
                                                           s.ctypes.data, None)
        assert status == 0, (name, dtype, _native.last_error())
        m0, u = int(s[2]), int(s[7])
        return {"plan": tuple(int(v) for v in s[:7]), "m0": m0, "u": u,
                "b": u * -(-m0 // u), "ctas": int(s[9])}

    f32 = {name: shape(name, _native.F32) for name in SPECIALISED_CASES}
    f64 = {name: shape(name, _native.F64) for name in SPECIALISED_CASES}
    # an unrolled block longer than the box (unaligned rows and time shards use this case)
    assert f32["cfg4 future"]["b"] != f32["cfg4 future"]["m0"], f32["cfg4 future"]
    assert f32["cfg4 future"]["u"] != f64["cfg4 future"]["u"]
    # three CTAs per SM, which float64 never gets (time shards, host pipeline, non-finite)
    assert f32["cfg2"]["ctas"] == 3 and f64["cfg2"]["ctas"] == 2
    assert all(s["ctas"] <= 2 for s in f64.values())
    # another plan than float64's: the planner's register bound depends on the element size
    for name in ("example default", "ecog-like"):
        assert f32[name]["plan"] != f64[name]["plan"], name
    # the short one-sided filter: the longest chunk in float32 (unaligned rows use it)
    assert f32["short future"]["u"] > f64["short future"]["u"]


def test_specialisation_threshold_grows_with_the_plan():
    """The job size from which the kernel is compiled for the plan (NVRTC: 0.5 s for the
    BASELINE tap sets, 22 s for 860 taps in runs of 41) scales with the square of the plan's
    unrolled work, so a cfg2-size job with a huge plan keeps the pre-built gather."""
    from pyparrm_b200 import _engine

    engine = _engine.DeviceEngine.__new__(_engine.DeviceEngine)  # no device needed for this
    base = _engine.DeviceEngine.SPECIALISE_FROM
    small = oracle.tap_offsets(2000 / 130 * (1 + 3e-6), 2000 / 130 / 50, 2000, 0, "both")
    huge = oracle.tap_offsets(30000 / 130, 20.0, 5000, 0, "past")
    assert engine._specialise_from(_native.plan_filter(small)[0]) == base
    assert engine._specialise_from(_native.plan_filter(huge)[0]) > 4 * 64 * 1_200_000
    assert engine._specialise_from(_native.plan_filter(huge, strategy=_native.PLAN_GATHER)[0]) == base

"""Record outputs of the UNMODIFIED reference as golden fixtures (tests/golden/).

TEST INFRASTRUCTURE; runs only in the build container, where the reference is
mounted read-only at /root/reference (see oracle/ref_shim.py).  Usage:

    python oracle/make_golden.py            # writes tests/golden/*.npz

What is recorded (all by calling the reference's own methods; nothing here
re-implements its arithmetic):

* ``example_dbs.npz``   bundled DBS recording (cfg1): every objective evaluation
  ``find_period()`` makes, per-run indices and candidate grids, the final period,
  the ``create_filter(2000, 20, "both", 0.01)`` filter and ``filter_data()``
  output, next to the shipped known answer ``matlab_filtered.npy``
  (examples/plot_use_parrm.py:43-45, 77-80, 135-141, 210-240).
* ``synthetic_2x30000.npz``  seeded synthetic recording (random-index branch of
  run 3): same captures, all three filter directions; the filtered outputs at the
  columns ``oracle.golden_inputs.sample_columns`` picks.
* ``ecog_lfp.npz``      bundled 2-channel ECoG/LFP recording: period + evaluations.
* ``taps.npz``          tap offsets and default half-widths for a parameter sweep.
* ``objective.npz``     ``_optimise_local`` values on seeded tiles.
* ``filter_edges.npz``  short / ragged inputs (T < filter length, foreign data); the inputs
  are not stored, only their sha256 (``oracle.golden_inputs.filter_edges_inputs``).

It also copies the four example ``.npy`` recordings into
``pyparrm_b200/data/example_data/`` (data files, not source) so that
``get_example_data_paths`` works in the drop-in.
"""

from __future__ import annotations

import os
import shutil
import sys
import time

import numpy as np
import scipy

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle.ref_shim import import_reference  # noqa: E402
from oracle.golden_inputs import (EDGE_FILTERS, EDGE_SHAPES, filter_edges_inputs,  # noqa: E402
                                   sample_columns, sha)
from pyparrm_b200.synthetic import make_recording  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")
DATA_DST = os.path.join(ROOT, "pyparrm_b200", "data", "example_data")


def store_filtered(out: dict, name: str, filtered: np.ndarray, taps: np.ndarray) -> None:
    """Keep ``filtered`` at the columns ``sample_columns`` picks (``<name>_filtered_cols``)."""
    cols = sample_columns(filtered.shape[1], taps)
    out[f"{name}_filtered_cols"] = cols
    out[f"{name}_filtered"] = np.ascontiguousarray(filtered[:, cols])


def meta() -> dict:
    return dict(
        numpy_version=np.__version__,
        scipy_version=scipy.__version__,
        reference="neuromodulation/PyPARRM 1.2.0dev (/root/reference)",
    )


class Recorder:
    """Wraps a reference PARRM instance's private seams to log what it computes."""

    def __init__(self, parrm):
        self.parrm = parrm
        self.calls = []  # (period, bandwidth, lambda, n_indices, value)
        self.indices = []
        self.grids = []
        self.estimates = []  # what each run's candidate grid was built around
        local = parrm._optimise_local
        centre = parrm._get_centre_indices
        grid = parrm._get_possible_periods

        def rec_local(period, data, indices, bandwidth, lambda_):
            value = local(period, data, indices, bandwidth, lambda_)
            self.calls.append(
                (float(np.asarray(period).ravel()[0]), int(bandwidth), float(lambda_),
                 int(indices.shape[0]), float(value))
            )
            return value

        def rec_centre(*a, **k):
            out = centre(*a, **k)
            self.indices.append(np.asarray(out).copy())
            return out

        def rec_grid(estimated_period, run):
            out = grid(estimated_period, run)
            self.grids.append(np.asarray(out).copy())
            self.estimates.append(np.asarray(estimated_period, dtype=np.float64))
            return out

        parrm._optimise_local = rec_local
        parrm._get_centre_indices = rec_centre
        parrm._get_possible_periods = rec_grid

    def pack(self) -> dict:
        calls = np.array(self.calls, dtype=np.float64).reshape(-1, 5)
        out = dict(calls=calls, n_runs=np.int64(len(self.indices)))
        for r, (idx, grid) in enumerate(zip(self.indices, self.grids)):
            out[f"run{r}_indices"] = idx.astype(np.int64)
            out[f"run{r}_periods"] = grid
            out[f"run{r}_estimate"] = self.estimates[r]
        return out


def taps_of(filt: np.ndarray) -> np.ndarray:
    hw = (filt.shape[0] - 1) // 2
    return (np.nonzero(filt < 0)[0] - hw).astype(np.int32)


def golden_example_dbs(ref):
    paths = ref.get_example_data_paths
    data = np.load(paths("example_data"))
    matlab = np.load(paths("matlab_filtered"))
    p = ref.PARRM(data=data, sampling_freq=200, artefact_freq=150, verbose=False)
    rec = Recorder(p)
    t0 = time.perf_counter()
    p.find_period()
    dt = time.perf_counter() - t0
    out = rec.pack()
    out["period"] = np.float64(p.period)
    out["find_period_seconds"] = np.float64(dt)
    p.create_filter(filter_half_width=2000, omit_n_samples=20,
                    filter_direction="both", period_half_width=0.01)
    out["filter"] = p.filter.copy()
    out["taps"] = taps_of(p.filter)
    out["filtered"] = p.filter_data().copy()
    out["matlab_filtered"] = matlab
    p.create_filter()  # all defaults
    out["default_half_width"] = np.int64(p._filter_half_width)
    out["default_period_half_width"] = np.float64(p._period_half_width)
    out["default_taps"] = taps_of(p.filter)
    out["default_filtered"] = p.filter_data().copy()
    out["data_sha256"] = sha(data)
    out.update(meta())
    np.savez_compressed(os.path.join(GOLDEN, "example_dbs.npz"), **out)
    print(f"example_dbs: period={p.period!r} evals={len(rec.calls)} {dt:.1f}s "
          f"max|ref-matlab|={np.abs(out['filtered'] - matlab).max():.2e}")


def golden_synthetic(ref):
    fs, fa = 2000, 130
    data = make_recording(2, 30000, fs, fa, seed=1)
    p = ref.PARRM(data=data, sampling_freq=fs, artefact_freq=fa, verbose=False)
    rec = Recorder(p)
    t0 = time.perf_counter()
    p.find_period(random_seed=0)
    dt = time.perf_counter() - t0
    out = rec.pack()
    out["period"] = np.float64(p.period)
    out["standard_data_sha256"] = sha(p._standard_data)
    for direction in ("both", "past", "future"):
        p.create_filter(filter_direction=direction)
        out[f"{direction}_taps"] = taps_of(p.filter)
        store_filtered(out, direction, p.filter_data(), out[f"{direction}_taps"])
    out["default_half_width"] = np.int64(p._filter_half_width)
    p.create_filter(filter_half_width=2000, omit_n_samples=3, filter_direction="both")
    out["hw2000_taps"] = taps_of(p.filter)
    store_filtered(out, "hw2000", p.filter_data(), out["hw2000_taps"])
    out["data_sha256"] = sha(data)
    out["recording"] = np.array([2, 30000, fs, fa, 1], dtype=np.int64)
    out.update(meta())
    np.savez_compressed(os.path.join(GOLDEN, "synthetic_2x30000.npz"), **out)
    print(f"synthetic: period={p.period!r} evals={len(rec.calls)} {dt:.1f}s")


def golden_ecog(ref):
    data = np.load(ref.get_example_data_paths("ecog_lfp_data"))
    # sampling / stimulation rates of examples/plot_example_dbs_data.py:46-47
    p = ref.PARRM(data=data, sampling_freq=1000, artefact_freq=130, verbose=False)
    rec = Recorder(p)
    t0 = time.perf_counter()
    p.find_period(random_seed=0)
    dt = time.perf_counter() - t0
    out = rec.pack()
    out["period"] = np.float64(p.period)
    out["data_sha256"] = sha(data)
    out["rates"] = np.array([1000.0, 130.0])
    out.update(meta())
    np.savez_compressed(os.path.join(GOLDEN, "ecog_lfp.npz"), **out)
    print(f"ecog_lfp: period={p.period!r} evals={len(rec.calls)} {dt:.1f}s")


def tap_parameter_sweep():
    """(period, phw (nan = default period/50), hw (-1 = default), omit, direction, n_samples)."""
    rows = []
    periods = [
        1.3311148014466094, 200 / 13, 200 / 13 * (1 + 3e-6), 200 / 29, 200 / 29 * (1 + 3e-6),
        3000 / 13, 3000 / 13 * (1 + 3e-6), 2.0, 2.0000001, 30.76923, 7.0, 6.896551724137931,
        15.384661538461538, 230.76992307692308, 1.5, 3.14159, 101.01, 0.75,
    ]
    for per in periods:
        # 2.0000001 never re-enters the `mod <= phw` band, so the default
        # half-width runs to (n - 1) // 2 (SURVEY S9); keep that case small.
        n_long = 20_000 if per == 2.0000001 else 1_200_000
        for direction in (0, 1, 2):
            rows.append((per, np.nan, -1, 0, direction, n_long))
            rows.append((per, np.nan, 2000, 0, direction, 1_200_000))
            rows.append((per, per / 50, 2000, 7, direction, 1_200_000))
        rows.append((per, per, 300, 0, 0, 100_000))          # every offset is a tap
        rows.append((per, per * 0.5, 301, 2, 0, 100_000))
        rows.append((per, 1e-6, 2000, 0, 0, 100_000))         # near-empty / empty
        rows.append((per, 0.01, 2000, 20, 0, 19_130))
        rows.append((per, np.nan, 10_000, 50, 0, 100_000))
        rows.append((per, np.nan, -1, 5, 0, 300))              # half-width capped by n
        rows.append((per, np.nan, 49, 48, 0, 100))             # test_parrm.py:291-294 shape
    return rows


def golden_taps(ref):
    directions = ("both", "past", "future")
    rows = tap_parameter_sweep()
    table, taps_flat, starts, default_hw = [], [], [0], []
    p = ref.PARRM(data=np.zeros((1, 8)), sampling_freq=1, artefact_freq=1, verbose=False)
    for per, phw, hw, omit, d, n in rows:
        per = float(per)
        phw_eff = per / 50 if np.isnan(phw) else float(phw)
        p._n_samples = int(n)
        p._period = np.float64(per)
        p._period_half_width = phw_eff
        p._omit_n_samples = int(omit)
        dhw = int(p._get_filter_half_width())
        hw_eff = dhw if hw < 0 else int(hw)
        p._filter_half_width = hw_eff
        p._filter_direction = directions[d]
        try:
            p._generate_filter()
            taps = taps_of(p._filter)
            n_taps = taps.shape[0]
            assert np.isclose(p._filter[p._filter < 0], -1.0 / n_taps).all()
        except RuntimeError:
            taps, n_taps = np.zeros(0, np.int32), -1
        table.append((per, phw_eff, hw_eff, omit, d, n, n_taps))
        default_hw.append(dhw)
        taps_flat.append(taps)
        starts.append(starts[-1] + taps.shape[0])
    np.savez_compressed(
        os.path.join(GOLDEN, "taps.npz"),
        table=np.array(table, dtype=np.float64),
        default_half_width=np.array(default_hw, dtype=np.int64),
        taps=np.concatenate(taps_flat).astype(np.int32),
        starts=np.array(starts, dtype=np.int64),
        **meta(),
    )
    print(f"taps: {len(rows)} parameter sets, {starts[-1]} taps, "
          f"{sum(1 for r in table if r[-1] < 0)} empty")


def golden_objective(ref):
    fs, fa = 2000, 130
    out = {}
    case = 0
    for n_chans in (1, 3):
        data = make_recording(n_chans, 30000, fs, fa, seed=2 + n_chans)
        p = ref.PARRM(data=data, sampling_freq=fs, artefact_freq=fa, verbose=False)
        p._outlier_boundary = 3.0
        p._standardise_data()
        z = p._standard_data
        rng = np.random.default_rng(7)
        index_sets = {
            "contig5001": np.arange(12499, 17500),
            "contig25001": np.arange(2499, 27500),
            "random": np.unique(rng.integers(0, 28000, 25000)) + 750,
        }
        p0 = fs / fa
        periods = np.concatenate((
            p0 * (1 + np.linspace(-1e-2, 1e-2, 9)),
            p0 * (1 + 3e-6) * (1 + np.linspace(-2e-5, 2e-5, 7)),
            [p0 / 2, p0 * 2, 9.87654321],
        ))
        for name, idx in index_sets.items():
            for bw, lam in ((5, 1.0), (10, 1.0), (20, 1.0), (20, 0.0)):
                if name == "contig5001" and bw == 20:
                    continue
                vals = np.array([p._optimise_local(per, z, idx, bw, lam) for per in periods])
                out[f"case{case}_indices"] = idx.astype(np.int64)
                out[f"case{case}_periods"] = periods
                out[f"case{case}_values"] = vals
                out[f"case{case}_params"] = np.array([n_chans, bw, lam, 2 + n_chans])
                case += 1
    out["n_cases"] = np.int64(case)
    out["recording"] = np.array([30000, fs, fa], dtype=np.int64)
    out.update(meta())
    np.savez_compressed(os.path.join(GOLDEN, "objective.npz"), **out)
    print(f"objective: {case} cases")


def golden_cfg2_objective(ref):
    """BASELINE cfg2 at full size (64 channels x 1.2 M samples): the reference's objective on
    the run-3 shape (random index branch, bandwidth 20) for 16 candidates of the run-3 grid
    spread over it, on all host threads (a whole find_period would take hours).  Also one
    channel's filtered output for the cfg2 filter, through the reference's filter_data."""
    from concurrent.futures import ThreadPoolExecutor

    fs, fa, n_chans, n = 2000, 130, 64, 1_200_000
    data = make_recording(n_chans, n, fs, fa, seed=0)
    p = ref.PARRM(data=data, sampling_freq=fs, artefact_freq=fa, verbose=False)
    p._search_samples = np.arange(n - 1)
    p._outlier_boundary = 3.0
    p._standardise_data()
    z = p._standard_data
    rng = np.random.default_rng(0)
    idx = [p._get_centre_indices(use_n, ignore, rng)
           for use_n, ignore in ((5000, 0.0), (10000, 0.0), (25000, 0.95))][-1]
    grid = p._get_possible_periods((fs / fa * (1 + 3e-6),), 3)
    pick = grid[np.linspace(0, len(grid) - 1, 16).astype(int)]
    with ThreadPoolExecutor(max_workers=os.cpu_count() or 1) as pool:
        vals = np.array(list(pool.map(lambda per: p._optimise_local(per, z, idx, 20, 1.0), pick)))
    out = dict(indices=idx.astype(np.int64), periods=pick, values=vals,
               recording=np.array([n_chans, n, fs, fa, 0], dtype=np.int64))
    q = ref.PARRM(data=data[:2], sampling_freq=fs, artefact_freq=fa, verbose=False)
    q._period = np.float64(fs / fa * (1 + 3e-6))
    q.create_filter(filter_half_width=2000, filter_direction="both")
    y = q.filter_data()
    out["filtered_ch1_head"] = y[1, :4000].copy()
    out["filtered_ch1_mid"] = y[1, 600000:602000].copy()
    out.update(meta())
    np.savez_compressed(os.path.join(GOLDEN, "cfg2_objective.npz"), **out)
    print(f"cfg2_objective: {len(pick)} candidates, {len(idx)} indices")


def golden_filter_edges(ref):
    out = {}
    xs = filter_edges_inputs()
    p = ref.PARRM(data=xs[0], sampling_freq=2000, artefact_freq=130, verbose=False)
    p._period = np.float64(2000 / 130 * (1 + 3e-6))
    case = 0
    for hw, omit, direction, phw in EDGE_FILTERS:
        p.create_filter(filter_half_width=hw, omit_n_samples=omit,
                        filter_direction=direction, period_half_width=phw)
        for _ in EDGE_SHAPES:
            x = xs[case]
            out[f"case{case}_x_sha256"] = sha(x)  # the tests regenerate x (oracle/golden_inputs.py)
            y = p.filter_data(x).copy()
            out[f"case{case}_y"] = y
            out[f"case{case}_taps"] = taps_of(p.filter)
            out[f"case{case}_hw"] = np.int64(hw)
            case += 1
    out["n_cases"] = np.int64(case)
    out.update(meta())
    np.savez_compressed(os.path.join(GOLDEN, "filter_edges.npz"), **out)
    print(f"filter_edges: {case} cases")


def golden_psd(ref):
    """compute_psd (src/pyparrm/_utils/_power.py:10-68) on seeded inputs: the reference
    function itself, imported from the unmodified package."""
    from pyparrm._utils._power import compute_psd

    rng = np.random.default_rng(44)
    out = {}
    cases = [  # shape, sampling_freq, n_points, max_freq
        ((2, 100), 20, 10, None), ((1, 100), 20, 10, 8.0), ((3, 5000), 1000, 200, 300.0),
        ((2, 300), 200, 1024, None), ((100,), 20, 16, None), ((4, 19130), 200, 40, 60.0),
        ((1, 20000), 2000, 4000, None),
    ]
    for k, (shape, fs, n, fmax) in enumerate(cases):
        x = rng.standard_normal(shape) * 3 + np.sin(np.arange(shape[-1]) * 0.7)
        freqs, psd = compute_psd(data=x, sampling_freq=fs, n_points=n, max_freq=fmax)
        if x.shape[-1] > 6000:  # only the first n_points samples matter: keep the fixture small
            x = np.ascontiguousarray(x[..., : n + 7])
            assert np.array_equal(compute_psd(data=x, sampling_freq=fs, n_points=n, max_freq=fmax)[1], psd)
        out[f"case{k}_x"] = x
        out[f"case{k}_args"] = np.array([fs, n, -1.0 if fmax is None else fmax])
        out[f"case{k}_freqs"] = freqs
        out[f"case{k}_psd"] = psd
    out["n_cases"] = np.int64(len(cases))
    out.update(meta())
    np.savez_compressed(os.path.join(GOLDEN, "psd.npz"), **out)
    print(f"psd: {len(cases)} cases")


def copy_example_recordings(ref):
    os.makedirs(DATA_DST, exist_ok=True)
    for name in ref.data.DATASETS:
        src = ref.get_example_data_paths(name)
        shutil.copyfile(src, os.path.join(DATA_DST, os.path.basename(src)))
    print(f"copied {len(ref.data.DATASETS)} example recordings")


def main():
    os.makedirs(GOLDEN, exist_ok=True)
    ref = import_reference()
    only = set(sys.argv[1:])
    jobs = dict(
        data=copy_example_recordings, taps=golden_taps, edges=golden_filter_edges,
        objective=golden_objective, example=golden_example_dbs,
        synthetic=golden_synthetic, ecog=golden_ecog, psd=golden_psd, cfg2=golden_cfg2_objective,
    )
    for name, job in jobs.items():
        if not only or name in only:
            job(ref)


if __name__ == "__main__":
    main()

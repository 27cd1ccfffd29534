"""``PARRM``: the reference's public class, with its two hot paths on a B200.

Drop-in for ``pyparrm.PARRM`` (reference ``src/pyparrm/parrm.py:18-936``): same constructor,
``find_period`` / ``create_filter`` / ``filter_data`` / ``explore_filter_params`` signatures,
same properties, same exception types and messages, same private attribute names (the
reference's own tests and its parameter explorer read them, ``tests/test_parrm.py:90-109``,
``_utils/_plotting.py:111-199``).  What changed is where the arithmetic runs:

===============================  =========================================================
reference (NumPy / SciPy, CPU)   here (hand-written sm_100a kernels behind a C ABI)
===============================  =========================================================
``_standardise_data`` :272-280   ``parrm_channel_scales`` + ``parrm_standardise_gather``
``_optimise_local`` :552-632     ``parrm_eval_periods`` (all candidates of a stage at once)
pqdm map over the grid :445-454  one batched launch per grid
5 x ``scipy fmin`` :499-517      lock-step Nelder-Mead, one batched launch per iteration
``_generate_filter`` :803-833    ``parrm_build_taps`` (integer-exact tap offsets)
``filter_data`` body :861-869    ``parrm_filter_apply`` (direct gather, no FFTs)
===============================  =========================================================

Host logic that decides *what* to evaluate (validation, index selection with NumPy's PCG64
stream, candidate grids, ranking, simplex moves, parameter defaults) stays in Python, as the
reference has it.  There is no CPU fallback for the arithmetic.
"""

from __future__ import annotations

from multiprocessing import cpu_count

import numpy as np

from . import _engine, _sharding
from ._neldermead import fmin_batch

np.seterr(all="ignore")  # the reference silences divide/invalid globally (parrm.py:15)

_SAMPLE_CAPS = (5000, 10000, 25000)      # parrm.py:291
_IGNORE_PORTIONS = (0.0, 0.0, 0.95)      # parrm.py:294
_BANDWIDTHS = (5, 10, 20)                # parrm.py:295
_GRID_LAMBDA = 1.0                       # parrm.py:296
_N_RESTARTS = 5                          # parrm.py:499
_HALF_WIDTH_MATCHES = 50                 # parrm.py:792
_DIRECTIONS = ["both", "past", "future"]  # parrm.py:781
_DEVICE_DTYPES = ("torch.float64", "torch.float32", "torch.int16", "torch.int32")

_NO_PERIOD_MSG = (
    "The period cannot be estimated from the data. Check that your data "
    "does not contain infs or NaNs."
)
_PERIOD_FIRST_MSG = (
    "The period has not yet been estimated. The `find_period` method must "
    "be called first."
)


def _require_number(value, name: str) -> None:
    if not isinstance(value, (int, float)):
        raise TypeError(f"`{name}` must be an int or a float.")


def _check_filter_out(out, data: np.ndarray, out_dtype) -> None:
    """Checks of ``filter_data(out=...)``: a writeable float64 / float32 array of the recording's
    shape, C-ordered or time-major, sharing no memory with it."""
    if not isinstance(out, np.ndarray):
        raise TypeError("`out` must be a NumPy array.")
    if out.shape != data.shape:
        raise ValueError(f"`out` must have the shape of `data` {data.shape}, not {out.shape}.")
    if out.dtype not in (np.dtype(np.float64), np.dtype(np.float32)):
        raise TypeError(f"`out` must be float64 or float32, not {out.dtype}.")
    if out_dtype is not None and np.dtype(out_dtype) != out.dtype:
        raise TypeError(f"`out_dtype` ({np.dtype(out_dtype)}) must match `out.dtype` ({out.dtype}).")
    if not out.flags.writeable:
        raise ValueError("`out` must be writeable.")
    if not out.flags.c_contiguous and _engine.time_major_ld(out) is None:
        raise ValueError("`out` must be C-contiguous or time-major (the transpose of a "
                         "[times, channels] array).")
    if np.may_share_memory(out, data):
        raise ValueError("`out` must not share memory with `data`.")


def _is_device_tensor(obj) -> bool:
    """True for a torch tensor that lives on a CUDA device (without importing torch here)."""
    return (type(obj).__module__.split(".")[0] == "torch" and hasattr(obj, "is_cuda")
            and bool(obj.is_cuda))


class PARRM:
    """Remove periodic stimulation artefacts with PARRM (Dastin-van Rijn et al., 2021).

    Call :meth:`find_period`, then :meth:`create_filter`, then :meth:`filter_data`.

    Parameters
    ----------
    data : numpy.ndarray, shape [channels, times]; or a CUDA ``torch.Tensor`` (additive)
        A CUDA tensor (float64 / float32, or int16 / int32 for ``filter_data()`` only) on the
        engine's GPU is searched and filtered where it lies: nothing crosses PCIe, and
        ``filter_data()`` / ``_standard_data`` are CUDA tensors.  ``find_period()`` gives
        bit for bit the period and fit errors of the NumPy array of the same values.
    sampling_freq, artefact_freq : int | float, in Hz
    verbose : bool (default True)
    precision : ``"fp64"`` (default, reference arithmetic) or ``"fp32"`` -- additive,
        keyword-only; ``"fp32"`` runs the filter kernel in single precision and keeps the
        search tiles in float32 (fit in float64); period and output within 1e-4 relative.
    """

    _data = None
    _standard_data_cache = None
    _filtered_data = None

    _sampling_freq = None
    _artefact_freq = None
    _verbose = None

    _period = None
    _search_samples = None
    _assumed_periods = None
    _outlier_boundary = None
    _random_seed = None
    _n_jobs = None

    _filter = None
    _filter_half_width = None
    _omit_n_samples = None
    _filter_direction = None
    _period_half_width = None

    _precision = "fp64"
    _standardised = False
    filter_shard = None  # (c0, c1, t0, t1) computed by this rank in the last filter_data()

    def __init__(self, data, sampling_freq, artefact_freq, verbose=True, *, precision="fp64"):
        self._check_init_inputs(data, sampling_freq, artefact_freq, verbose)
        if precision not in ("fp64", "fp32"):
            raise ValueError("`precision` must be 'fp64' or 'fp32'.")
        self._precision = precision
        self._n_chans, self._n_samples = self._data.shape

    # ------------------------------------------------------------------ inputs
    def _check_init_inputs(self, data, sampling_freq, artefact_freq, verbose) -> None:
        """Constructor checks (reference parrm.py:112-140), plus CUDA-tensor recordings."""
        if _is_device_tensor(data):
            if str(data.dtype) not in _DEVICE_DTYPES:
                raise TypeError(
                    f"A CUDA tensor `data` must be float64, float32, int16 or int32, not "
                    f"{data.dtype}.")
            device = getattr(_engine.get_engine(), "device", None)
            if device is not None and data.device != device:
                raise ValueError(
                    f"`data` is on {data.device}, but this process computes on {device}.")
        elif not isinstance(data, np.ndarray):
            raise TypeError("`data` must be a NumPy array.")
        if data.ndim != 2:
            raise ValueError("`data` must be a 2D array.")
        self._data = data  # held by reference, never modified

        _require_number(sampling_freq, "sampling_freq")
        if sampling_freq <= 0:
            raise ValueError("`sampling_freq` must be > 0.")
        self._sampling_freq = sampling_freq

        _require_number(artefact_freq, "artefact_freq")
        if artefact_freq <= 0:
            raise ValueError("`artefact_freq` must be > 0.")
        self._artefact_freq = artefact_freq

        if not isinstance(verbose, bool):
            raise TypeError("`verbose` must be a bool.")
        self._verbose = verbose

    def __repr__(self) -> str:
        return (
            f"PARRM object | Data: ({self._n_chans} channels x "
            f"{self._n_samples} times) | Period: {self._period:.4f}"
        )

    # ------------------------------------------------------------- period search
    def find_period(
        self,
        search_samples=None,
        assumed_periods=None,
        outlier_boundary=3.0,
        random_seed=None,
        n_jobs=1,
    ) -> None:
        """Find the period of the artefacts (reference parrm.py:148-194).

        ``n_jobs`` is validated exactly as in the reference and otherwise ignored: every
        candidate of a stage is evaluated in one GPU launch.
        """
        if self._verbose:
            print("\nFinding the artefact period...")
        if _sharding.active() and _is_device_tensor(self._data):
            raise NotImplementedError(
                "find_period() on a CUDA-tensor recording does not shard: the tensor belongs to "
                "this rank alone, and the sharded search needs the same recording on every "
                "rank. Call disable_sharding() first, or pass a NumPy array.")
        self._reset_result_attrs()
        self._check_sort_find_stim_period_inputs(
            search_samples, assumed_periods, outlier_boundary, random_seed, n_jobs
        )
        self._standardise_data()
        self._optimise_period_estimate()
        if self._verbose:
            print("    ... Artefact period found\n")

    def _reset_result_attrs(self) -> None:
        """Forget everything derived from a previous period (reference parrm.py:196-211)."""
        self._standard_data_cache = None
        self._standardised = False
        self._filtered_data = None
        self._period = None
        self._search_samples = None
        self._assumed_periods = None
        self._outlier_boundary = None
        self._random_seed = None
        self._filter = None
        self._filter_half_width = None
        self._omit_n_samples = None
        self._filter_direction = None
        self._period_half_width = None

    def _check_sort_find_stim_period_inputs(
        self, search_samples, assumed_periods, outlier_boundary, random_seed, n_jobs
    ) -> None:
        """``find_period`` argument checks and defaults (reference parrm.py:213-270)."""
        if search_samples is not None and not isinstance(search_samples, np.ndarray):
            raise TypeError("`search_samples` must be a NumPy array or None.")
        if search_samples is None:
            # the default range is sorted as it is made (the reference sorts it all the same:
            # 9 ms of a 46 ms search on a 1.2 M-sample recording)
            search_samples = np.arange(self._n_samples - 1)
        elif search_samples.ndim != 1:
            raise ValueError("`search_samples` must be a 1D array.")
        else:
            search_samples = np.sort(search_samples)
        if search_samples[0] < 0 or search_samples[-1] >= self._n_samples:
            raise ValueError(
                "Entries of `search_samples` must lie in the range [0, n_samples)."
            )
        self._search_samples = search_samples

        if assumed_periods is not None and not isinstance(assumed_periods, (int, float, tuple)):
            raise TypeError("`assumed_periods` must be an int, a float, a tuple, or None.")
        if assumed_periods is None:
            assumed_periods = (self._sampling_freq / self._artefact_freq,)
        elif isinstance(assumed_periods, (int, float)):
            assumed_periods = (assumed_periods,)
        elif not all(isinstance(entry, (int, float)) for entry in assumed_periods):
            raise TypeError("If a tuple, entries of `assumed_periods` must be ints or floats.")
        self._assumed_periods = assumed_periods

        _require_number(outlier_boundary, "outlier_boundary")
        if outlier_boundary <= 0:
            raise ValueError("`outlier_boundary` must be > 0.")
        self._outlier_boundary = outlier_boundary

        if random_seed is not None and not isinstance(random_seed, int):
            raise TypeError("`random_seed` must be an int or None.")
        if random_seed is not None:
            self._random_seed = random_seed

        if not isinstance(n_jobs, int):
            raise TypeError("`n_jobs` must be an int.")
        if n_jobs > cpu_count():
            raise ValueError("`n_jobs` must be <= the number of available CPUs.")
        if n_jobs <= 0 and n_jobs != -1:
            raise ValueError("If `n_jobs` is <= 0, it must be -1.")
        self._n_jobs = cpu_count() if n_jobs == -1 else n_jobs

    def _standardise_data(self) -> None:
        """Reference parrm.py:272-280.  Deferred: the device computes the per-channel scale
        and gathers only the fitted columns (``DeviceEngine.prepare_tiles``); the full
        ``[channels, times - 1]`` array is materialised only if ``_standard_data`` is read."""
        if _is_device_tensor(self._data):
            floating = self._data.is_floating_point()
        else:
            floating = np.issubdtype(self._data.dtype, np.floating)
        if not floating:
            # NumPy refuses the in-place true divide on an integer difference
            raise TypeError(
                "Cannot standardise non-floating data in place "
                f"(dtype {self._data.dtype}); pass float64 or float32 data."
            )
        self._standardised = True
        self._standard_data_cache = None

    @property
    def _standard_data(self):
        if self._standardised and self._standard_data_cache is None:
            self._standard_data_cache = _engine.get_engine().standardise_full(
                self._data, self._outlier_boundary
            )
        return self._standard_data_cache

    @_standard_data.setter
    def _standard_data(self, value) -> None:
        self._standard_data_cache = value
        self._standardised = value is not None

    def _optimise_period_estimate(self) -> None:
        """Coarse-to-fine period search (reference parrm.py:282-325)."""
        engine = _engine.get_engine()
        random_state = np.random.default_rng(self._random_seed)

        sample_lens = np.unique(
            [int(np.min((self._search_samples.shape[0], cap))) for cap in _SAMPLE_CAPS]
        )
        plan = list(zip(sample_lens, _IGNORE_PORTIONS, _BANDWIDTHS))
        # Index sets depend only on the search range and the RNG stream, never on the data,
        # so all runs' sets are drawn up front (same draw order as the reference) and the
        # recording crosses PCIe once.
        index_sets = [
            self._get_centre_indices(use_n, ignore, random_state) for use_n, ignore, _ in plan
        ]
        if _sharding.active():  # every rank standardises its channel block; tiles all-gathered
            tiles = _sharding.prepare_tiles_sharded(
                engine, self._data, index_sets, self._outlier_boundary, self._precision)
        else:
            tiles = engine.prepare_tiles(self._data, index_sets, self._outlier_boundary,
                                         self._precision)

        estimated_period = self._assumed_periods
        for run_idx, ((_, _, bandwidth), indices, tile) in enumerate(
            zip(plan, index_sets, tiles), start=1
        ):
            bandwidth = int(np.min((bandwidth, indices.shape[0] // 4)))
            periods = self._get_possible_periods(estimated_period, run_idx)
            periods, fit_errors = self._optimise_period_estimate_first_run(
                periods, tile, bandwidth, _GRID_LAMBDA
            )
            estimated_period = self._optimise_period_estimate_second_run(
                periods, fit_errors, tile, bandwidth, _GRID_LAMBDA
            )

        if not np.isfinite(estimated_period[0]):
            raise ValueError(_NO_PERIOD_MSG)

        # last run's samples, unclamped last bandwidth, no regularisation (parrm.py:323-325)
        self._period = self._optimise_period_estimate_final_run(
            estimated_period[0], tiles[-1], _BANDWIDTHS[-1]
        )

    def _get_centre_indices(self, use_n_samples, ignore_portion, random_state) -> np.ndarray:
        """Samples fitted in one run (reference parrm.py:327-374): a window centred on the
        search range or, when that range is much longer, sorted unique random draws from its
        middle ``1 - ignore_portion``."""
        first, last = self._search_samples[0], self._search_samples[-1]
        centre_sum = first + last
        lo = int(np.ceil((centre_sum - use_n_samples) / 2))
        hi = int(np.floor((centre_sum + use_n_samples) / 2))
        if self._n_samples * ignore_portion < hi - lo:
            return np.arange(lo, hi + 1)

        margin = (1.0 - ignore_portion) / 2.0 * self._n_samples
        lo = int(first + np.floor(margin))
        hi = int(last - np.ceil(margin))
        draws = random_state.integers(0, hi - lo, np.min((use_n_samples, hi - lo)))
        return np.unique(draws) + lo

    def _get_possible_periods(self, estimated_period, run: int) -> np.ndarray:
        """Candidate periods around each estimate (reference parrm.py:376-405): +-1 % in
        steps of 1e-4 and +-0.1 % in steps of 1e-5, both shrunk by the run number."""
        relative = np.concatenate(
            (
                (1 + np.arange(-1e-2, 1e-2 + 1e-4, 1e-4) / run),
                (1 + np.arange(-1e-3, 1e-3 + 1e-5, 1e-5) / run),
            )
        )
        candidates = []
        for period in estimated_period:
            candidates.extend(period * relative)
        return np.unique(candidates)

    def _evaluate(self, periods, tile, bandwidth, lambda_) -> np.ndarray:
        return _engine.get_engine().evaluate(tile, periods, bandwidth, lambda_, self._n_chans)

    def _evaluate_grid(self, periods, tile, bandwidth, lambda_) -> np.ndarray:
        """The data-parallel map of the reference (pqdm, parrm.py:445-454).  Under
        ``pyparrm_b200.enable_sharding()`` the candidates are split over the ranks and the fit
        errors exchanged with one all-gather."""
        if _sharding.active():
            engine = _engine.get_engine()
            # device engine: the block's errors stay on the GPU through the all-gather
            evaluate = getattr(engine, "evaluate_device", engine.evaluate)
            return _sharding.evaluate_sharded(
                lambda block: evaluate(tile, block, bandwidth, lambda_, self._n_chans), periods
            )
        return self._evaluate(periods, tile, bandwidth, lambda_)

    def _fmin(self, starts, tile, bandwidth, lambda_):
        """``scipy.optimize.fmin`` at its defaults from each start (parrm.py:499-517, 545-550):
        on the device engine the simplex state machines run on the GPU with the rounds replayed
        as CUDA graphs (``DeviceEngine.nm_minimise``); any other engine drives the same state
        machines from the host (``_neldermead.fmin_batch``)."""
        engine = _engine.get_engine()
        if hasattr(engine, "nm_minimise"):
            return engine.nm_minimise(tile, starts, bandwidth, lambda_, self._n_chans)
        return fmin_batch(lambda p: self._evaluate(p, tile, bandwidth, lambda_), starts)

    def _optimise_period_estimate_first_run(self, periods, tile, bandwidth, lambda_):
        """Evaluate the grid and rank it (reference parrm.py:407-465)."""
        fit_error = self._evaluate_grid(periods, tile, bandwidth, lambda_)
        order = fit_error.argsort()
        fit_error = fit_error[order]
        periods = periods[order[np.isfinite(fit_error)]]
        if periods.shape == (0,):
            raise ValueError(_NO_PERIOD_MSG)
        return periods, fit_error

    def _optimise_period_estimate_second_run(self, periods, fit_errors, tile, bandwidth, lambda_):
        """Nelder-Mead from the best five candidates (reference parrm.py:467-522)."""
        n_iters = int(np.min((_N_RESTARTS, periods.shape[0])))
        results = self._fmin(periods[:n_iters], tile, bandwidth, lambda_)
        for k, (x, fval, _, _) in enumerate(results):
            periods[k] = x
            fit_errors[k] = fval
        return (periods[fit_errors.argmin()],)

    def _optimise_period_estimate_final_run(self, period, tile, bandwidth):
        """Unregularised polish of the final estimate (reference parrm.py:524-550)."""
        return self._fmin([period], tile, bandwidth, 0.0)[0][0]

    def _optimise_local(self, period, data, indices, bandwidth, lambda_) -> float:
        """Fit error for one period (the reference's evaluator seam, parrm.py:552-597).

        ``data`` is an already standardised ``[channels, times]`` array.  Kept for callers that
        drive the evaluator directly; ``find_period`` itself batches candidates instead."""
        engine = _engine.get_engine()
        tile = engine.tile_from_standardised(np.asarray(data), np.asarray(indices))
        value = engine.evaluate(
            tile, np.atleast_1d(np.asarray(period, dtype=np.float64)), int(bandwidth),
            float(lambda_), self._n_chans,
        )
        return value[0]

    # ----------------------------------------------------------- explorer (GUI)
    def explore_filter_params(
        self, time_range=None, time_res=0.01, freq_range=None, freq_res=5.0, n_jobs=1
    ) -> None:
        """Interactive parameter explorer (reference parrm.py:634-687).

        The matplotlib GUI is outside the accelerated path and is not shipped; the entry point
        keeps the reference's precondition and then reports that."""
        if self._verbose:
            print("Opening the filter parameter explorer...")
        if self._period is None:
            raise ValueError(_PERIOD_FIRST_MSG)
        raise NotImplementedError(
            "pyparrm_b200 accelerates find_period / create_filter / filter_data; the "
            "matplotlib parameter explorer of the reference is not part of this build."
        )

    # ------------------------------------------------------------------- filter
    def create_filter(
        self,
        filter_half_width=None,
        omit_n_samples=0,
        filter_direction="both",
        period_half_width=None,
    ) -> None:
        """Create the PARRM filter (reference parrm.py:689-737)."""
        if self._verbose:
            print("Creating the filter...")
        if self._period is None:
            raise ValueError(_PERIOD_FIRST_MSG)
        self._check_sort_create_filter_inputs(
            filter_half_width, omit_n_samples, filter_direction, period_half_width
        )
        self._generate_filter()
        if self._verbose:
            print("    ... Filter created\n")

    def _check_sort_create_filter_inputs(
        self, filter_half_width, omit_n_samples, filter_direction, period_half_width
    ) -> None:
        """``create_filter`` argument checks and defaults, in the reference's order
        (parrm.py:739-786): omit -> period half-width -> filter half-width -> direction."""
        half_span = (self._n_samples - 1) // 2

        if not isinstance(omit_n_samples, int):
            raise TypeError("`omit_n_samples` must be an int.")
        if omit_n_samples < 0 or omit_n_samples >= half_span:
            raise ValueError(
                "`omit_n_samples` must lie in the range [0, (no. of samples - 1) // 2)."
            )
        self._omit_n_samples = omit_n_samples

        if period_half_width is None:
            period_half_width = self._period / 50
        _require_number(period_half_width, "period_half_width")
        if period_half_width <= 0 or period_half_width > self._period:
            raise ValueError("`period_half_width` must be lie in the range (0, period].")
        self._period_half_width = period_half_width

        if filter_half_width is None:
            filter_half_width = self._get_filter_half_width()
        if not isinstance(filter_half_width, int):
            raise TypeError("`filter_half_width` must be an int.")
        if filter_half_width <= omit_n_samples or filter_half_width > half_span:
            raise ValueError(
                "`filter_half_width` must lie in the range (`omit_n_samples`, "
                "(no. of samples - 1) // 2]."
            )
        self._filter_half_width = filter_half_width

        if not isinstance(filter_direction, str):
            raise TypeError("`filter_direction` must be a str.")
        if filter_direction not in _DIRECTIONS:
            raise ValueError(f"`filter_direction` must be one of {_DIRECTIONS}.")
        self._filter_direction = filter_direction

    def _get_filter_half_width(self) -> int:
        """Default half-width: the first that holds 50 phase-matched offsets past the omitted
        ones, capped at ``(n - 1) // 2`` (reference parrm.py:788-801).  The reference's second
        clause compares against ``period + half_width`` and so never fires; kept as is.
        Vectorised in blocks; visits offsets in the same order as the reference's loop."""
        limit = (self._n_samples - 1) // 2
        start = self._omit_n_samples
        needed = _HALF_WIDTH_MATCHES
        block = 4096
        while start < limit:
            offsets = np.arange(start + 1, min(start + block, limit) + 1)
            phase = np.mod(offsets, self._period)
            hit = (phase <= self._period_half_width) | (
                phase >= self._period + self._period_half_width
            )
            running = np.cumsum(hit)
            if running[-1] >= needed:
                return int(offsets[np.searchsorted(running, needed)])
            needed -= int(running[-1])
            start = int(offsets[-1])
            block = min(block * 4, 1 << 22)
        return int(max(start, self._omit_n_samples))

    def _generate_filter(self) -> None:
        """Build ``self._filter`` (reference parrm.py:803-833): taps get ``-1 / n_taps``, the
        centre 1.  The tap offsets come from the device tap builder (bit-exact with the
        reference's NumPy mask)."""
        half_width = self._filter_half_width
        taps = _engine.get_engine().build_taps(
            self._period, self._period_half_width, half_width, self._omit_n_samples,
            self._filter_direction,
        )
        if taps.shape[0] == 0:
            raise RuntimeError(
                "A suitable filter cannot be created with the specified settings. Try "
                "reducing the number of omitted samples and/or increasing the filter "
                "half-width."
            )
        filter_ = np.zeros(2 * half_width + 1, dtype=np.float64)
        filter_[taps.astype(np.int64) + half_width] = 1.0
        filter_ = -filter_ / np.max((filter_.sum(), np.finfo(filter_.dtype).eps))
        filter_[half_width] = 1
        self._filter = filter_

    def filter_data(self, data=None, *, out_dtype=None, out=None) -> np.ndarray:
        """Apply the PARRM filter and return the result (reference parrm.py:835-875).

        Output is float64 ``[channels, times]`` (``out_dtype=numpy.float32``, keyword-only and
        additive, halves the bytes that come back over PCIe).  float32 / int16 / int32
        recordings are uploaded in their own width and widened on the device.  Where no tap falls inside the recording
        (first / last samples of a one-sided filter) the result is 0, the documented intent of
        parrm.py:867-869 (the reference's FFT path returns rounding noise there).

        ``data`` may also be a CUDA ``torch.Tensor`` ``[channels, times]`` (additive): it is
        filtered where it lies and a device tensor comes back -- nothing crosses PCIe (and
        nothing is sharded: under ``enable_sharding()`` the tensor is this rank's own).  So is
        the object's own recording when that is a CUDA tensor and ``data`` is not given.

        Under ``pyparrm_b200.enable_sharding()`` every rank filters its channel block (time
        block when channels are fewer than ranks, halos read from the recording); what comes
        back follows the ``gather`` mode given there, and ``filter_shard`` holds the
        ``(c0, c1, t0, t1)`` range this rank computed.

        Time-major recordings -- ``mm.T`` or ``mm[:, a:b].T`` of a ``[times, channels]`` array
        such as ``np.load("run.npy", mmap_mode="r")``, the layout SpikeGLX / Open Ephys / Intan
        files hold -- are read as they lie and transposed on the device: no host copy is made.

        ``out`` (keyword-only, additive, NumPy recordings only): a writeable float64 / float32
        ``[channels, times]`` array to fill and return instead of a new one -- C-ordered, or
        time-major such as ``np.lib.format.open_memmap(path, "w+", np.float32, (T, C)).T``, which
        writes the result in the file's own layout.  It must not share memory with ``data``;
        ``out_dtype``, if given, must be ``out.dtype``."""
        if self._verbose:
            print("Filtering the data...")
        if self._filter is None:
            raise ValueError(
                "The filter has not yet been created. The `create_filter` method must "
                "be called first."
            )
        taps = self._tap_offsets()
        engine = _engine.get_engine()
        if data is None and _is_device_tensor(self._data):
            data = self._data  # a CUDA recording is filtered where it lies, as below
        if _is_device_tensor(data):
            # additive overload (SURVEY 8(f).2): a CUDA tensor [channels, times] (float64 or
            # float32) is filtered where it lies and the result stays on the device -- no PCIe
            # in either direction; `filtered_data` then holds the device tensor
            if data.dim() != 2:
                raise ValueError("`data` must be a 2D array.")
            if out_dtype is not None:
                raise TypeError("`out_dtype` applies to NumPy results; convert the returned tensor.")
            if out is not None:
                raise TypeError("`out` applies to NumPy recordings; a CUDA tensor is filtered "
                                "into a new device tensor.")
            d_x = data if data.stride(1) == 1 else data.contiguous()
            want = engine.torch.float32 if self._precision == "fp32" else engine.torch.float64
            if d_x.dtype != want:  # float32 / integer recordings are widened, as on the host path
                d_x = d_x.to(want)
            self.filter_shard = (0, d_x.shape[0], 0, d_x.shape[1])
            self._filtered_data = engine.filter_device(d_x, taps)
            if self._verbose:
                print("    ... Data filtered\n")
            return self._filtered_data
        data = self._check_sort_filter_data_inputs(data)
        if out is not None:
            if _sharding.active():
                raise NotImplementedError(
                    "filter_data(out=...) does not shard: call disable_sharding() first, or "
                    "let filter_data() return its result.")
            _check_filter_out(out, data, out_dtype)
        if _sharding.active():
            result, self.filter_shard, _ = _sharding.filter_sharded(
                engine, data, taps, self._precision, _sharding.gather_mode(), out_dtype)
            self._filtered_data = result
        else:
            self.filter_shard = (0, data.shape[0], 0, data.shape[1])
            extra = {} if out is None else {"out": out}
            self._filtered_data = engine.filter_host(data, taps, self._precision,
                                                     out_dtype=out_dtype, **extra)
        if self._verbose:
            print("    ... Data filtered\n")
        return self._filtered_data

    def _tap_offsets(self) -> np.ndarray:
        """Ascending offsets ``w`` of the filter's taps (``y[t]`` reads ``x[t - w]``)."""
        half_width = (self._filter.shape[0] - 1) // 2
        return (np.flatnonzero(self._filter < 0) - half_width).astype(np.int32)

    def filter_stream(self, *, max_chunk=1 << 16, out_dtype=None, graphs=False, history=0):
        """Filter a recording block by block as it is acquired (additive).

        Returns a :class:`pyparrm_b200._stream.FilterStream` holding a snapshot of this
        object's filter and precision (a later ``create_filter()`` does not affect it)::

            parrm.find_period(); parrm.create_filter(filter_direction="future")
            stream = parrm.filter_stream()
            for block in acquisition:     # [channels, n] NumPy array or CUDA tensor
                y = stream.push(block)    # [channels, k]: every output that is now final
            tail = stream.close()         # the last `stream.latency` outputs

        The pushes and ``close()`` concatenate to exactly ``filter_data()`` of the concatenated
        recording.  Output ``t`` is final once sample ``t + stream.latency`` has arrived;
        ``latency = max(0, -min(taps))`` is 0 for ``filter_direction="future"``, the causal
        direction (``y[t]`` reads ``x[t - w]``, and its taps ``w`` are positive), and
        ``filter_half_width`` at most for ``"past"`` and ``"both"``.

        ``max_chunk``: the longest push the device ring is sized for (longer pushes are split
        on the host).  ``out_dtype``: float64 (default) or float32 NumPy results; CUDA-tensor
        pushes return CUDA tensors in the compute type.  ``graphs=True`` replays NumPy pushes of a
        repeated shape as one CUDA graph (H2D, kernel, D2H); the results are the same bit for
        bit, but on a B200 it measured 8-18 us slower per push than the default separate
        launches (profiles/r3/stream_latency.txt).  Not available under ``enable_sharding()``.

        ``history``: samples per channel the stream keeps on the device for
        ``stream.recent(n)``, ``n <= history``, so that the filter can be re-calibrated from the
        stream's own recent samples and switched in with ``stream.set_filter(cal)``::

            stream = parrm.filter_stream(history=10 * fs)    # keep the last 10 s on the device
            for block in acquisition:
                y = stream.push(block)
                if settings_changed:                        # e.g. a new stimulation frequency
                    cal = PARRM(stream.recent(10 * fs), fs, new_fa, verbose=False)
                    cal.find_period()                       # on the GPU, no PCIe
                    cal.create_filter(filter_half_width=hw, filter_direction="future")
                    stream.set_filter(cal)                  # outputs not yet returned: new taps

        ``create_filter()`` bounds ``filter_half_width`` by ``(n - 1) // 2`` of the window it was
        calibrated on, so the window must hold at least ``2 * filter_half_width + 1`` samples.
        The ring then holds ``max(span, history) + max_chunk`` samples per channel; with
        ``history=0`` (default) it, the launches and the push times are as without it."""
        if self._filter is None:
            raise ValueError(
                "The filter has not yet been created. The `create_filter` method must "
                "be called first."
            )
        if _sharding.active():
            raise NotImplementedError(
                "filter_stream() does not shard: a stream runs on this rank's GPU only. Call "
                "disable_sharding() first, or filter whole recordings with filter_data()."
            )
        from ._stream import FilterStream

        return FilterStream(_engine.get_engine(), self._tap_offsets(), self._precision,
                            max_chunk=max_chunk, out_dtype=out_dtype, graphs=graphs,
                            history=history)

    def filter_sweep(self, parameter_sets, data=None):
        """Filter with many parameter sets at once (additive; SURVEY 8(f).4).

        ``parameter_sets``: iterable of dicts with the keyword arguments of
        :meth:`create_filter` (``filter_half_width``, ``omit_n_samples``, ``filter_direction``,
        ``period_half_width``; missing keys take ``create_filter``'s defaults, validated with
        the same rules and messages).  The default half-widths of all sets come from one
        launch, all tap sets from one launch and all filtered copies from one launch -- what
        the reference's explorer does with one ``_generate_filter`` + ``filter_data`` per
        widget event (``_utils/_plotting.py:568-584``).  Returns ``(filtered, taps)``:
        float64 ``[n_sets, channels, times]`` and the list of tap-offset arrays.  Leaves the
        object's own filter untouched."""
        if self._period is None:
            raise ValueError(_PERIOD_FIRST_MSG)
        data = self._check_sort_filter_data_inputs(data)
        engine = _engine.get_engine()
        half_span = (self._n_samples - 1) // 2
        sets = [dict(s) for s in parameter_sets]
        omits, phws, hws, dirs = [], [], [], []
        for s in sets:
            omit = s.get("omit_n_samples", 0)
            if not isinstance(omit, int):
                raise TypeError("`omit_n_samples` must be an int.")
            if omit < 0 or omit >= half_span:
                raise ValueError(
                    "`omit_n_samples` must lie in the range [0, (no. of samples - 1) // 2).")
            phw = s.get("period_half_width")
            if phw is None:
                phw = self._period / 50
            _require_number(phw, "period_half_width")
            if phw <= 0 or phw > self._period:
                raise ValueError("`period_half_width` must be lie in the range (0, period].")
            direction = s.get("filter_direction", "both")
            if not isinstance(direction, str):
                raise TypeError("`filter_direction` must be a str.")
            if direction not in _DIRECTIONS:
                raise ValueError(f"`filter_direction` must be one of {_DIRECTIONS}.")
            omits.append(omit), phws.append(float(phw)), dirs.append(direction)
            hws.append(s.get("filter_half_width"))
        missing = [i for i, hw in enumerate(hws) if hw is None]
        if missing:  # parrm.py:788-801 for every set that asked for the default, one launch
            found = engine.default_half_widths(
                [self._period] * len(missing), [phws[i] for i in missing],
                [omits[i] for i in missing], half_span)
            for i, hw in zip(missing, found):
                hws[i] = int(hw)
        for hw, omit in zip(hws, omits):
            if not isinstance(hw, int):
                raise TypeError("`filter_half_width` must be an int.")
            if hw <= omit or hw > half_span:
                raise ValueError(
                    "`filter_half_width` must lie in the range (`omit_n_samples`, "
                    "(no. of samples - 1) // 2].")
        return engine.filter_sweep(data, [float(self._period)] * len(sets), phws, hws, omits, dirs)

    def _check_sort_filter_data_inputs(self, data) -> np.ndarray:
        """Reference parrm.py:877-886."""
        if data is None:
            data = self._data
        if not isinstance(data, np.ndarray):
            raise TypeError("`data` must be a NumPy array.")
        if data.ndim != 2:
            raise ValueError("`data` must be a 2D array.")
        return data

    # --------------------------------------------------------------- properties
    @property
    def data(self) -> np.ndarray:
        return self._data

    @property
    def period(self) -> float:
        if self._period is None:
            raise AttributeError("No period has been computed yet.")
        return self._period

    @property
    def filter(self) -> np.ndarray:
        if self._filter is None:
            raise AttributeError("No filter has been computed yet.")
        return self._filter

    @property
    def filtered_data(self) -> np.ndarray:
        if self._filtered_data is None:
            raise AttributeError("No data has been filtered yet.")
        return self._filtered_data

    @property
    def settings(self) -> dict:
        """Settings used to generate the filter (reference parrm.py:914-936)."""
        if self._period is None or self._filter is None:
            raise AttributeError("Analysis settings have not been established yet.")
        return {
            "data": {
                "sampling_freq": self._sampling_freq,
                "artefact_freq": self._artefact_freq,
            },
            "period": {
                "search_samples": self._search_samples,
                "assumed_periods": self._assumed_periods,
                "outlier_boundary": self._outlier_boundary,
                "random_seed": self._random_seed,
            },
            "filter": {
                "filter_half_width": self._filter_half_width,
                "omit_n_samples": self._omit_n_samples,
                "filter_direction": self._filter_direction,
                "period_half_width": self._period_half_width,
            },
        }

#!/usr/bin/env python
"""Benchmark of the PARRM hot paths on B200: ``python bench.py --gpus N --steps K --warmup W``.

Headline (BASELINE.json ``metric``): ``filter_data`` channel-samples/s on configs[1] --
synthetic 64-channel LFP, 2 kHz, 130 Hz stimulation artefact, 10 min (64 x 1 200 000 float64),
``create_filter(filter_half_width=2000, filter_direction="both")`` (160 taps).  One *step* is
one pass of the filter over the whole recording.

* ``value``  -- recording resident in HBM, one ``parrm_filter_apply`` launch per step, timed with
  CUDA events on the launching stream (inputs are 614 MB, larger than the 126 MB L2).
* ``e2e``    -- the same pass through the public API ``PARRM.filter_data()`` with a pinned host
  array in and a host array out: H2D + kernel + D2H inside the timed region every step.
* ``roofline`` -- 16 algorithmic bytes per channel-sample (8 read + 8 written) / kernel time,
  against the measured HBM copy bandwidth in MEASURED_PEAKS.json.
* ``cpu_baseline`` -- the UNMODIFIED reference (``oracle/_ref``, a verbatim copy made by
  ``oracle/vendor_ref.py``, imported through the dispatch-only shims of ``oracle/ref_shim.py``)
  running ``PARRM.filter_data()`` on all 64 channels of the same recording, on this host.
* ``find_period`` -- second metric of BASELINE.json: candidate periods/s of the evaluator on
  the same recording (run-3 shape: ~24.7 k random samples x 64 channels, 20 harmonics, the
  388-candidate grid), with its FP64-pipe roofline and the reference's ``_optimise_local`` on
  all host threads beside it (plus a labelled non-reference process-parallel line).
* ``e2e_variants`` -- the same API call with a pageable array, with the caller's array
  registered in place, and with float32 in / float32 out (half the PCIe bytes).
* ``cfg1`` -- BASELINE configs[0]: find_period + create_filter + filter_data on the bundled
  example recording, wall time here and for the reference on this host.
* ``strong`` -- strong-scaling cases: cfg4 (384 channels x 9 M samples, one-sided filter,
  channel-sharded) and a cfg5 candidate sweep (1e5 periods, winner by one (error, index)
  pair per rank).

``--steps K`` is the number of timed passes of ``value``, ``e2e`` (per window), each
``e2e_variants`` window and ``find_period`` (its fp32 mode too); the strong-scaling,
``standardise`` and power-capped (``roofline.sustained``) figures time fixed counts of their own.

``--impl reference`` times the unmodified reference's ``PARRM.filter_data()`` on this host's
cores on bounded samples of the same workload; rank 0 only; it maps no library of this repo.

``--dump-outputs DIR`` (rank 0) writes, after the timed steps, what the last of them computed:
``filter_data.npy``, rows ``DUMP_ROWS`` of the headline's filtered recording (float64
[4, 1 200 000]), and ``find_period_errors.npy``, the evaluator's fit errors of its last timed
step (float64).  The inputs are seeded, so two builds run with the same arguments can be
compared output for output.

Multi-GPU (torchrun, one rank per GPU) goes through the product's own sharding API:
``pyparrm_b200.enable_sharding()`` + ``PARRM.filter_data()`` / ``PARRM.find_period()``.  Weak
scaling for the headline: the recording grows to N x 64 channels, channel-sharded, no
collective; the period search shards the candidate grid and all-gathers the errors over NCCL.
"""

from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_CHANS, N_SAMPLES, FS, FA = 64, 1_200_000, 2000, 130
HALF_WIDTH = 2000
WORKLOAD = ("cfg2: synthetic 64-ch LFP, 2 kHz, 130 Hz DBS artefact, 10 min (64 x 1.2M f64), "
            "filter_half_width=2000, bidirectional")
BYTES_PER_CHANNEL_SAMPLE = 16.0  # float64: 8 read + 8 written (SURVEY 8(d))
# --dump-outputs keeps these whole rows of the 614 MB filtered recording (38.4 MB): every
# sample of a row, the edges included, where the taps run off the recording
DUMP_ROWS = np.sort(np.random.default_rng(0).choice(N_CHANS, 4, replace=False))
DUMP_LIMIT_BYTES = 64 << 20


# ----------------------------------------------------------------------------- helpers
def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            peaks = json.load(fh)
        return float(peaks["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """Samples SM clock and throttle reasons through NVML while the timed regions run."""

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self.period = 0.002
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _loop(self):
        nv = self.nv
        names = {
            "hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
            "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
            "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
            "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4),
            "hw_power_brake": getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80),
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
                for name, bit in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(self.period)

    def __enter__(self):
        if self.nv is not None:
            self._thread = threading.Thread(target=self._loop, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        if self._thread is not None:
            self._thread.join()

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml unavailable"]}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def dist_setup(n_gpus: int):
    import torch

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist

        torch.cuda.set_device(local)
        # before any pinned allocation: keep this rank's host buffers on its GPU's NUMA node
        from pyparrm_b200._sharding import bind_host_to_gpu

        bind_host_to_gpu(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        return dist, world, rank, local
    torch.cuda.set_device(0)
    return None, 1, 0, 0


def max_over_ranks(dist, seconds: float) -> float:
    if dist is None:
        return seconds
    import torch

    t = torch.tensor([seconds], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def all_ranks(dist, value: float) -> list:
    """The value of every rank, in rank order (diagnostic: which GPU set the max)."""
    if dist is None:
        return [value]
    import torch

    mine = torch.tensor([value], dtype=torch.float64, device="cuda")
    every = torch.empty(dist.get_world_size(), dtype=torch.float64, device="cuda")
    dist.all_gather_into_tensor(every, mine)
    return [float(v) for v in every.cpu()]


def barrier(dist):
    import torch

    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()


def dump_outputs(directory: str, arrays: dict) -> None:
    """Write each array as ``directory/<name>.npy``, so that two builds can be compared output
    for output on the same seeded inputs."""
    nbytes = sum(a.nbytes for a in arrays.values())
    if nbytes > DUMP_LIMIT_BYTES:
        raise ValueError(f"--dump-outputs: {nbytes} bytes, more than {DUMP_LIMIT_BYTES}")
    for name, array in arrays.items():
        if array.dtype not in (np.float32, np.float64):
            raise TypeError(f"--dump-outputs: {name} is {array.dtype}, not float32 or float64")
    for name, array in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), array)


# ----------------------------------------------------------------------------- CPU legs
def import_reference():
    """The unmodified reference package (oracle/_ref or /root/reference), or None."""
    from oracle import ref_shim

    if not ref_shim.reference_available():
        return None, "reference neither mounted nor vendored (python oracle/vendor_ref.py)"
    return ref_shim.import_reference(), ref_shim.reference_location()


def reference_filter_object(pyparrm, data, period):
    """Reference PARRM object with the benchmark's filter, period injected (the filter
    benchmark does not depend on the search)."""
    ref = pyparrm.PARRM(data, FS, FA, verbose=False)
    ref._period = np.float64(period)
    ref.create_filter(filter_half_width=HALF_WIDTH, filter_direction="both")
    return ref


def cpu_filter_baseline(data, period):
    """Reference filter_data() on the whole recording, one pass (single-threaded by design:
    scipy.signal.convolve, parrm.py:861-866)."""
    pyparrm, where = import_reference()
    if pyparrm is None:
        from oracle import parrm_oracle as oracle

        filt = oracle.build_filter(period, period / 50, HALF_WIDTH, 0, "both")
        t0 = time.perf_counter()
        oracle.apply_filter_fft(data, filt)
        seconds = time.perf_counter() - t0
        kind, what = "port", f"oracle port ({where})"
    else:
        ref = reference_filter_object(pyparrm, data, period)
        t0 = time.perf_counter()
        ref.filter_data()
        seconds = time.perf_counter() - t0
        kind, what = "reference", f"unmodified reference PARRM.filter_data() from {where}"
    line = {
        "value": data.size / seconds, "unit": "channel-samples/s", "cores": 1, "kind": kind,
        "sample": f"all {data.shape[0]} channels x {data.shape[1]} samples, 1 pass, {seconds:.1f} s; "
                  f"{what}; single-threaded as the reference runs it",
    }
    try:  # best-effort CPU line, NOT the reference's execution model: channels over processes
        from joblib import Parallel, delayed

        from oracle import parrm_oracle as oracle

        filt = oracle.build_filter(period, period / 50, HALF_WIDTH, 0, "both")
        workers = min(os.cpu_count() or 1, data.shape[0])
        blocks = np.array_split(np.arange(data.shape[0]), workers)
        # start the workers (and their SciPy import) outside the timed pass
        Parallel(n_jobs=workers)(delayed(oracle.apply_filter_fft)(data[:1, :4096], filt)
                                 for _ in range(2 * workers))
        t0 = time.perf_counter()
        Parallel(n_jobs=workers)(delayed(oracle.apply_filter_fft)(data[b], filt) for b in blocks)
        par_seconds = time.perf_counter() - t0
        line["non_reference_process_parallel"] = {
            "value": data.size / par_seconds, "unit": "channel-samples/s", "cores": workers,
            "what": f"joblib processes over channel blocks, oracle port of parrm.py:861-869 (the same "
                    f"two FFT convolutions), {par_seconds:.2f} s with warm workers, including "
                    "shipping the blocks both ways"}
    except Exception as err:  # noqa: BLE001
        line["non_reference_process_parallel"] = {"unavailable": str(err)[:100]}
    return line


def cpu_search_baseline(data, indices, periods, bandwidth, n_candidates=None):
    """Reference _optimise_local over grid candidates on all host threads (the pqdm.threads map
    of parrm.py:445-454), plus a labelled NON-reference process-parallel line (joblib)."""
    from oracle import parrm_oracle as oracle

    cores = os.cpu_count() or 1
    n_candidates = n_candidates or max(cores, 16)
    z = oracle.standardise(data, 3.0)
    pick = periods[np.linspace(0, len(periods) - 1, n_candidates).astype(int)]
    pyparrm, where = import_reference()
    if pyparrm is not None:
        from concurrent.futures import ThreadPoolExecutor

        ref = pyparrm.PARRM(data, FS, FA, verbose=False)
        t0 = time.perf_counter()
        with ThreadPoolExecutor(max_workers=cores) as pool:
            list(pool.map(lambda p: ref._optimise_local(p, z, indices, bandwidth, 1.0), pick))
        seconds = time.perf_counter() - t0
        kind, what = "reference", f"unmodified reference PARRM._optimise_local from {where}"
    else:
        t0 = time.perf_counter()
        oracle.objective_many(pick, z, indices, bandwidth, 1.0, data.shape[0], n_jobs=cores)
        seconds = time.perf_counter() - t0
        kind, what = "port", "oracle port"
    line = {
        "value": n_candidates / seconds, "unit": "candidates/s", "cores": cores, "kind": kind,
        "sample": f"{n_candidates} of {len(periods)} grid candidates x {len(indices)} samples x "
                  f"{data.shape[0]} channels, bw={bandwidth}, {cores} threads (pqdm.threads "
                  f"equivalent), {seconds:.1f} s; {what}",
    }
    try:  # best-effort CPU line, NOT the reference's execution model (SURVEY 8(d))
        from joblib import Parallel, delayed

        workers = min(cores, n_candidates)
        t0 = time.perf_counter()
        Parallel(n_jobs=workers)(delayed(oracle.objective)(p, z, indices, bandwidth, 1.0,
                                                           data.shape[0]) for p in pick)
        seconds = time.perf_counter() - t0
        line["non_reference_process_parallel"] = {
            "value": n_candidates / seconds, "unit": "candidates/s", "cores": workers,
            "what": f"joblib processes over candidates, oracle port of the objective, {seconds:.1f} s "
                    "(includes shipping the standardised recording to the workers)"}
    except Exception as err:  # noqa: BLE001
        line["non_reference_process_parallel"] = {"unavailable": str(err)[:100]}
    return line


# ----------------------------------------------------------------------------- reference arm
def run_reference(args):
    """Times the unmodified reference.  Imports nothing that maps libparrm_b200.so."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from pyparrm_b200.synthetic import make_recording, true_period  # pure NumPy module

    period = true_period(FS, FA)
    pyparrm, where = import_reference()
    probe = make_recording(2, N_SAMPLES, FS, FA, seed=0)
    if pyparrm is not None:
        run_pass = lambda obj: obj.filter_data()  # noqa: E731
        make = lambda d: reference_filter_object(pyparrm, d, period)  # noqa: E731
        kind = "reference"
        what = f"unmodified reference PARRM.filter_data() (parrm.py:835-875) from {where}"
    else:
        from oracle import parrm_oracle as oracle

        filt = oracle.build_filter(period, period / 50, HALF_WIDTH, 0, "both")
        run_pass = lambda d: oracle.apply_filter_fft(d, filt)  # noqa: E731
        make = lambda d: d  # noqa: E731
        kind, what = "port", f"oracle port of parrm.py:861-869 ({where})"
    t0 = time.perf_counter()
    run_pass(make(probe))
    per_chan = (time.perf_counter() - t0) / 2
    budget = 170.0
    n_chans = int(max(1, min(N_CHANS, budget / ((args.steps + args.warmup) * per_chan))))
    sample = make_recording(n_chans, N_SAMPLES, FS, FA, seed=0)
    obj = make(sample)
    for _ in range(args.warmup):
        run_pass(obj)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        run_pass(obj)
    seconds = time.perf_counter() - t0
    value = sample.size * args.steps / seconds
    line = {
        "impl": "reference", "metric": "filter_data channel-samples/sec", "value": value,
        "unit": "channel-samples/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * seconds / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": WORKLOAD, "taps": 160, "sharding": "CPU, rank 0 only",
                   "l2": "n/a (CPU)", "timing": "host wall clock (CPU path)"},
        "cpu_baseline": {
            "value": value, "unit": "channel-samples/s", "cores": 1, "kind": kind,
            "sample": f"{n_chans} of {N_CHANS} channels x {N_SAMPLES} samples per step (as many "
                      f"channels as fit {budget:.0f} s for {args.steps}+{args.warmup} steps; the rate "
                      f"per channel does not depend on the count); {what}; scipy.signal.convolve "
                      "(FFT), single-threaded as the reference runs it",
        },
        "e2e": {"value": value, "unit": "channel-samples/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- B200 arm
def recorded_pcie_floor(n_gpus: int):
    """Bare concurrent pinned H2D + D2H of one cfg2 pass per GPU, N ranks at once, as recorded
    by scripts/pcie_rate.py on an earlier box (profiles/r2/pcie_floor.jsonl) -- context for the
    e2e figure, not measured in this run."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2", "pcie_floor.jsonl")) as fh:
            for line in fh:
                if line.startswith("{"):
                    rec = json.loads(line)
                    if rec.get("n_gpus") == n_gpus:
                        return {"ms_per_step": rec["h2d_d2h_concurrent"]["ms"],
                                "value": rec["e2e_floor_channel_samples_per_s"],
                                "source": "profiles/r2/pcie_floor.jsonl (scripts/pcie_rate.py under "
                                          "torchrun, recorded earlier on another box of this pool)"}
    except Exception:
        pass
    return None


def timed_api_passes(dist, fn, steps):
    import torch

    barrier(dist)
    t0 = time.perf_counter()
    marks = [t0]
    for _ in range(steps):
        out = fn()
        marks.append(time.perf_counter())
    torch.cuda.synchronize()
    seconds = max_over_ranks(dist, time.perf_counter() - t0)
    barrier(dist)
    timed_api_passes.last_pass_ms = [round(1e3 * (b - a), 2) for a, b in zip(marks, marks[1:])]
    return seconds, out


def run_b200(args):
    import torch

    from oracle import parrm_oracle as oracle  # cpu legs and the parity guard only
    from pyparrm_b200 import (PARRM, _engine, _sharding, disable_sharding, enable_sharding,
                              pin_array, pinned_empty)
    from pyparrm_b200.synthetic import make_recording, true_period

    dist, world, rank, local = dist_setup(args.gpus)
    engine = _engine.get_engine()
    hbm_peak, peak_source = measured_peaks()
    period = true_period(FS, FA)
    units = N_CHANS * N_SAMPLES

    # The job: one recording of world x 64 channels (weak scaling), channel-sharded by the
    # product's own plan.  Every rank materialises only its rows of the host array (the other
    # rows are never touched: PARRM holds `data` by reference and a rank reads its shard only).
    total_chans = world * N_CHANS
    if world > 1:
        enable_sharding(gather="none")
        recording = np.empty((total_chans, N_SAMPLES), dtype=np.float64)
    else:
        recording = pinned_empty((total_chans, N_SAMPLES))
    parrm = PARRM(recording, FS, FA, verbose=False)
    parrm._period = np.float64(period)
    parrm.create_filter(filter_half_width=HALF_WIDTH, filter_direction="both")
    taps = (np.flatnonzero(parrm.filter < 0) - HALF_WIDTH).astype(np.int32)
    w_lo, w_hi = min(int(taps[0]), 0), max(int(taps[-1]), 0)
    c0, c1, t0_, t1_, _, _ = _sharding.channel_or_time_shards(total_chans, N_SAMPLES, world,
                                                              w_lo, w_hi)[rank]
    assert (c1 - c0, t0_, t1_) == (N_CHANS, 0, N_SAMPLES)
    data = recording[c0:c1]
    make_recording(N_CHANS, N_SAMPLES, FS, FA, seed=rank, out=data)
    pin = pin_array(data) if world > 1 else None  # in place: only this rank's rows are locked

    d_x = torch.from_numpy(data).cuda()
    d_y = torch.empty_like(d_x)
    stream = torch.cuda.current_stream()

    with ClockSampler(local) as clocks:
        # ---- value: device resident -------------------------------------------------
        for _ in range(args.warmup):
            engine.filter_device(d_x, taps, d_out=d_y)
        # A pass is 0.25 ms: W passes are over before a GPU that idled at the rendezvous is at
        # its boost clocks (ranks that waited ran 0.28-0.29 ms per pass for the whole region,
        # the others 0.255), while 50 ms or more of back-to-back passes put the GPU at its power
        # cap (0.265-0.275 ms; scripts/warmup_sweep.py: 2-20 ms of warm-up give 0.2475).  So:
        # rendezvous, 10 ms of passes with every rank in step, rendezvous again (immediate),
        # then the timed region -- the burst condition the measured HBM peak was taken under.
        # The power-capped rate is measured separately below (roofline.sustained).
        barrier(dist)
        for _ in range(40):
            engine.filter_device(d_x, taps, d_out=d_y)
        torch.cuda.synchronize()
        barrier(dist)
        launches0 = engine.launches
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record(stream)
        for _ in range(args.steps):
            engine.filter_device(d_x, taps, d_out=d_y)
        stop.record(stream)
        barrier(dist)
        launches = engine.launches - launches0
        filter_kernel = engine.last_filter_kernel
        dev_seconds = max_over_ranks(dist, start.elapsed_time(stop) * 1e-3)
        kernel_seconds = start.elapsed_time(stop) * 1e-3 / args.steps  # one launch per step
        rank_ms = [round(1e3 * v, 4) for v in all_ranks(dist, kernel_seconds)]
        dumped = {}
        if args.dump_outputs and rank == 0:
            dumped["filter_data"] = d_y[DUMP_ROWS.tolist()].cpu().numpy()

        # the same pass after half a second of back-to-back passes: the GPU at its power cap
        t_hot = time.perf_counter()
        while time.perf_counter() - t_hot < 0.5:
            for _ in range(40):
                engine.filter_device(d_x, taps, d_out=d_y)
            torch.cuda.synchronize()
        h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        h0.record(stream)
        for _ in range(50):
            engine.filter_device(d_x, taps, d_out=d_y)
        h1.record(stream)
        torch.cuda.synchronize()
        sustained_seconds = max_over_ranks(dist, h0.elapsed_time(h1) * 1e-3 / 50)

        standardise = bench_standardise(engine, d_x, hbm_peak) if world == 1 else None

        # ---- e2e: public API, host in / host out (sharded through enable_sharding) ---
        for _ in range(min(args.warmup, 3)):
            parrm.filter_data()
        # back-to-back windows of --steps passes, all reported; the line's e2e is the fastest
        # one.  The path is bound by the host's PCIe / memory system, which this process shares
        # with whatever else runs on the box, so windows repeat -- at most five -- until the two
        # fastest agree within 3 %.  (A result kept alive across windows makes the next window
        # page-lock a third 614 MB result buffer, ~0.5 s once: the [14.2, 40.3, 14.2] ms pattern
        # of earlier runs.  The previous result is dropped first.)
        e2e_windows, e2e_passes = [], []
        out = None
        for _ in range(5):
            out = None
            seconds, out = timed_api_passes(dist, parrm.filter_data, args.steps)
            e2e_windows.append(seconds)
            e2e_passes.append(timed_api_passes.last_pass_ms)
            best = sorted(e2e_windows)
            if len(best) >= 2 and best[1] <= 1.03 * best[0]:
                break
        e2e_seconds = min(e2e_windows)
        assert tuple(parrm.filter_shard) == (c0, c1, 0, N_SAMPLES)

        # ---- find_period evaluator (second metric) + the sharded search API ----------
        search = bench_search(engine, dist, world, rank, args, dumped)

        # ---- strong-scaling cases (device resident) --------------------------------
        strong = bench_strong(engine, dist, world, rank)

    # parity guard on what was just timed (3 channels against the oracle's direct form)
    want = oracle.apply_filter_direct(data[:3], taps)
    parity = float(np.abs(out[:3] - want).max() / np.abs(data[:3]).max())
    assert parity <= 1e-9, f"bench parity check failed: {parity:.3e}"
    dev_parity = float(np.abs(d_y[:3].cpu().numpy() - want).max() / np.abs(data[:3]).max())
    assert dev_parity <= 1e-9, f"bench parity check (device path) failed: {dev_parity:.3e}"

    variants, cfg1 = {}, None
    if world == 1:
        variants = bench_e2e_variants(engine, data, taps, args.steps, period)
        cfg1 = bench_cfg1(engine)
    if pin is not None:
        pin.release()
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dumped)

    cpu = cpu_filter_baseline(data, period) if world == 1 else None
    achieved = BYTES_PER_CHANNEL_SAMPLE * units / kernel_seconds / 1e9
    traffic = None
    try:
        with open(os.path.join(ROOT, "profiles", "filter_traffic.json")) as fh:
            traffic = json.load(fh).get("dram_bytes_per_launch")
    except Exception:
        pass
    line = {
        "metric": "filter_data channel-samples/sec",
        "value": world * units * args.steps / dev_seconds,
        "unit": "channel-samples/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * dev_seconds / args.steps,
        "ms_per_step_by_rank": rank_ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {
            "workload": WORKLOAD, "taps": int(taps.shape[0]),
            "sharding": (f"pyparrm_b200.enable_sharding(gather='none') + PARRM.filter_data() on one "
                         f"[{total_chans} x {N_SAMPLES}] recording: channel shards of 64 per GPU, "
                         "no collective" if world > 1 else "single GPU"),
            "l2": "inputs (614 MB/GPU) larger than L2 (126 MB); no flush needed",
            "timing": "CUDA events on the launching stream, max over ranks",
        },
        "clocks": clocks.summary(),
        "e2e": {
            "value": world * units * args.steps / e2e_seconds, "unit": "channel-samples/s",
            "h2d_bytes_per_step": units * 8, "d2h_bytes_per_step": units * 8,
            "steps": args.steps, "ms_per_step": 1e3 * e2e_seconds / args.steps,
            "windows_ms_per_step": [round(1e3 * w / args.steps, 3) for w in e2e_windows],
            "slowest_window_pass_ms": e2e_passes[int(np.argmax(e2e_windows))],
            "pcie_floor": recorded_pcie_floor(world),
            "api": ("PARRM.filter_data() under enable_sharding(gather='none'); this rank's rows "
                    "page-locked in place with pin_array()" if world > 1 else
                    "PARRM.filter_data() on a pinned NumPy array, NumPy result"),
        },
        "gpu_launches": launches,
        "roofline": {
            "bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
            "frac": achieved / hbm_peak, "traffic": traffic,
            "kernel": filter_kernel, "peak_source": peak_source,
            "algorithmic_bytes_per_launch": BYTES_PER_CHANNEL_SAMPLE * units,
            "sustained": {
                "ms_per_step": 1e3 * sustained_seconds,
                "frac": BYTES_PER_CHANNEL_SAMPLE * units / sustained_seconds / 1e9 / hbm_peak,
                "what": "the same launch after 0.5 s of back-to-back passes (GPU at its power cap: "
                        "sw_power_cap), max over ranks, against the same burst copy peak",
            },
        },
        "parity_max_rel_err": max(parity, dev_parity),
        "find_period": search,
        "strong": strong,
    }
    if standardise is not None:
        line["standardise"] = standardise
    if cpu is not None:
        line["cpu_baseline"] = cpu
    if variants:
        line["e2e_variants"] = variants
    if cfg1 is not None:
        line["cfg1"] = cfg1
    print(json.dumps(line), flush=True)
    if dist is not None:
        disable_sharding()
        dist.destroy_process_group()


def bench_standardise(engine, d_x, hbm_peak):
    """Row a1 (_standardise_data, parrm.py:272-280) on the device-resident recording: the
    streaming mean|diff| reduction reads every sample once (8 B per channel-sample)."""
    import torch

    from pyparrm_b200 import _native
    from pyparrm_b200._engine import _vp

    n_chans, n_samples = d_x.shape
    lib = _native.lib
    ws_bytes = lib.parrm_channel_scales_workspace_bytes(n_chans, n_samples)
    ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device="cuda")
    scale = torch.empty(n_chans, dtype=torch.float64, device="cuda")
    stream = torch.cuda.current_stream()
    sp = _vp(stream.cuda_stream)

    def once():
        _native.check(lib.parrm_channel_scales(_vp(d_x.data_ptr()), n_chans, n_samples, n_samples,
                                               _vp(scale.data_ptr()), _vp(ws.data_ptr()), ws_bytes,
                                               _native.F64, sp), "parrm_channel_scales")

    for _ in range(3):
        once()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 20
    e0.record(stream)
    for _ in range(reps):
        once()
    e1.record(stream)
    torch.cuda.synchronize()
    seconds = e0.elapsed_time(e1) * 1e-3 / reps
    achieved = 8.0 * n_chans * n_samples / seconds / 1e9
    return {"kernel": "abs_diff_partial_kernel + scale_finalise_kernel (parrm_channel_scales)",
            "ms": 1e3 * seconds, "value": n_chans * n_samples / seconds, "unit": "channel-samples/s",
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                         "frac": achieved / hbm_peak,
                         "algorithmic_bytes_per_launch": 8.0 * n_chans * n_samples}}


def bench_e2e_variants(engine, data, taps, steps, period):
    """The API call as existing callers make it (pageable np.ndarray), with the caller's array
    registered in place, and with half the PCIe bytes (float32 in, float32 out)."""
    import torch

    from pyparrm_b200 import PARRM, pin_array

    def rate(array, **kw):
        p = PARRM(array, FS, FA, verbose=False)
        p._period = np.float64(period)
        p.create_filter(filter_half_width=HALF_WIDTH, filter_direction="both")
        for _ in range(2):
            p.filter_data(**kw)
        windows = []
        for _ in range(2):  # two windows, the faster one reported (host-bound: noisy)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(steps):
                p.filter_data(**kw)
            torch.cuda.synchronize()
            windows.append(time.perf_counter() - t0)
        seconds = min(windows)
        return {"value": array.size * steps / seconds, "unit": "channel-samples/s",
                "ms_per_step": 1e3 * seconds / steps,
                "windows_ms_per_step": [round(1e3 * w / steps, 2) for w in windows]}

    out = {}
    pageable = np.array(data)  # ordinary malloc'ed copy, as np.load would hand over
    out["pageable_f64"] = dict(rate(pageable), h2d_bytes_per_step=data.size * 8,
                               d2h_bytes_per_step=data.size * 8,
                               what="pageable float64 in (staged through pinned buffers by "
                                    "parrm_host_copy, 8 threads), float64 out")
    t0 = time.perf_counter()
    handle = pin_array(pageable)
    register_ms = 1e3 * (time.perf_counter() - t0)
    out["registered_f64"] = dict(rate(pageable), register_ms=register_ms,
                                 what="same array after pyparrm_b200.pin_array(data) "
                                      "(cudaHostRegister once, direct copies afterwards)")
    handle.release()
    x32 = pageable.astype(np.float32)
    h32 = pin_array(x32)
    out["f32_in_f32_out"] = dict(rate(x32, out_dtype=np.float32), h2d_bytes_per_step=data.size * 4,
                                 d2h_bytes_per_step=data.size * 4,
                                 what="float32 recording uploaded as float32, widened on the device, "
                                      "float64 arithmetic, filter_data(out_dtype=float32)")
    h32.release()
    return out


def bench_cfg1(engine):
    """BASELINE configs[0]: the bundled example recording, whole workflow."""
    import torch

    from pyparrm_b200 import PARRM, get_example_data_paths

    data = np.load(get_example_data_paths("example_data"))

    def workflow(cls):
        p = cls(data, 200, 150, verbose=False)
        p.find_period()
        p.create_filter(filter_half_width=2000, omit_n_samples=20, filter_direction="both",
                        period_half_width=0.01)
        return p, p.filter_data()

    workflow(PARRM)  # builds / loads kernels
    torch.cuda.synchronize()
    launches0 = engine.launches
    t0 = time.perf_counter()
    p, out = workflow(PARRM)
    torch.cuda.synchronize()
    gpu_seconds = time.perf_counter() - t0
    result = {"workload": "cfg1: bundled example DBS recording (1 x 19130, 200 Hz / 150 Hz): "
                          "find_period() + create_filter(2000, 20, 'both', 0.01) + filter_data()",
              "gpu_seconds": gpu_seconds, "gpu_launches": engine.launches - launches0,
              "period": float(p.period)}
    pyparrm, where = import_reference()
    if pyparrm is not None:
        t0 = time.perf_counter()
        ref, ref_out = workflow(pyparrm.PARRM)
        result["reference_seconds"] = time.perf_counter() - t0
        result["reference_period"] = float(ref.period)
        result["period_equal"] = bool(ref.period == p.period)
        result["filtered_max_abs_diff"] = float(np.abs(ref_out - out).max())
        result["reference"] = f"unmodified reference from {where}, n_jobs=1 (its default)"
    return result


def bench_strong(engine, dist, world, rank):
    """Strong scaling, device resident: total work fixed, split by the product's plan."""
    import torch

    from oracle import parrm_oracle as oracle  # tap list of the named filter only
    from pyparrm_b200 import _sharding

    out = {}
    # ---- cfg4: 384 channels x 9 M samples (30 kHz x 300 s), one-sided filter ------------
    n_chans, n_samples, fs, fa, hw = 384, 9_000_000, 30000, 130, 2311
    per4 = fs / fa * (1 + 3e-6)
    taps = oracle.tap_offsets(per4, per4 / 50, hw, 0, "past")
    c0, c1, _, _, _, _ = _sharding.channel_or_time_shards(
        n_chans, n_samples, world, min(int(taps[0]), 0), max(int(taps[-1]), 0))[rank]
    gen = torch.Generator(device="cuda").manual_seed(100 + rank)
    d_x = torch.randn((c1 - c0, n_samples), dtype=torch.float64, device="cuda", generator=gen)
    d_y = torch.empty_like(d_x)
    for _ in range(2):
        engine.filter_device(d_x, taps, d_out=d_y)
    barrier(dist)
    steps = 5
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    stream = torch.cuda.current_stream()
    start.record(stream)
    for _ in range(steps):
        engine.filter_device(d_x, taps, d_out=d_y)
    stop.record(stream)
    barrier(dist)
    mine = start.elapsed_time(stop) * 1e-3
    seconds = max_over_ranks(dist, mine)
    hbm_peak, _ = measured_peaks()
    # spot parity at full size: one channel's window against the oracle's direct sum
    lo = 4_000_000
    xs = d_x[0, lo - 3000: lo + 8000].cpu().numpy()[None, :]
    ys = d_y[0, lo: lo + 5000].cpu().numpy()
    ref = oracle.apply_filter_direct(xs, taps)[0, 3000:8000]
    spot = float(np.abs(ys - ref).max() / np.abs(xs).max())
    assert spot <= 1e-9, f"cfg4 spot parity {spot:.3e}"
    out["cfg4_filter"] = {
        "workload": "cfg4: 384 ch x 9.0 M samples f64 (27.6 GB), 130 Hz at 30 kHz, one-sided "
                    f"('past') default-width filter, {len(taps)} taps; channel-sharded {c1 - c0} per GPU",
        "value": n_chans * n_samples * steps / seconds, "unit": "channel-samples/s",
        "ms_per_step": 1e3 * seconds / steps, "scaling": "strong",
        "kernel": engine.last_filter_kernel,
        "roofline_frac_this_rank": 16.0 * (c1 - c0) * n_samples * steps / mine / 1e9 / hbm_peak,
        "spot_parity_rel_err": spot,
    }
    del d_x, d_y
    # ---- cfg3 at full size on one GPU (256 ch x 3.6 M, 198 taps): roofline only ----------
    if world == 1:
        per3 = 1000 / 145 * (1 + 3e-6)
        taps3 = oracle.tap_offsets(per3, per3 / 50, 2469, 0, "both")
        d_x = torch.randn((256, 3_600_000), dtype=torch.float64, device="cuda", generator=gen)
        d_y = torch.empty_like(d_x)
        for _ in range(2):
            engine.filter_device(d_x, taps3, d_out=d_y)
        start.record(stream)
        for _ in range(steps):
            engine.filter_device(d_x, taps3, d_out=d_y)
        stop.record(stream)
        torch.cuda.synchronize()
        sec3 = start.elapsed_time(stop) * 1e-3
        out["cfg3_filter"] = {
            "workload": f"cfg3: 256 ch x 3.6 M samples f64 (7.4 GB), 145 Hz at 1 kHz, default "
                        f"half-width 2469, {len(taps3)} taps",
            "value": 256 * 3_600_000 * steps / sec3, "unit": "channel-samples/s",
            "ms_per_step": 1e3 * sec3 / steps, "kernel": engine.last_filter_kernel,
            "roofline_frac": 16.0 * 256 * 3_600_000 * steps / sec3 / 1e9 / hbm_peak,
        }
        del d_x, d_y
        # ---- float32 mode of the filter (PARRM(precision="fp32")), cfg2 shape -----------
        per2 = FS / FA * (1 + 3e-6)
        taps2 = oracle.tap_offsets(per2, per2 / 50, HALF_WIDTH, 0, "both")
        d_x = torch.randn((N_CHANS, N_SAMPLES), dtype=torch.float32, device="cuda", generator=gen)
        d_y = torch.empty_like(d_x)
        for _ in range(3):
            engine.filter_device(d_x, taps2, d_out=d_y)
        steps32 = 20
        start.record(stream)
        for _ in range(steps32):
            engine.filter_device(d_x, taps2, d_out=d_y)
        stop.record(stream)
        torch.cuda.synchronize()
        sec32 = start.elapsed_time(stop) * 1e-3
        xs = d_x[0, :30_000].double().cpu().numpy()[None, :]
        ref = oracle.apply_filter_direct(xs, taps2)[0, 5000:25_000]
        err32 = float(np.abs(d_y[0, 5000:25_000].cpu().numpy() - ref).max() / np.abs(xs).max())
        assert err32 <= 1e-4, f"float32 mode parity {err32:.3e}"
        out["cfg2_filter_fp32_mode"] = {
            "workload": "cfg2 shape, float32 storage and arithmetic (precision='fp32'; tolerance "
                        "1e-4 of the input scale against the float64 oracle)",
            "value": N_CHANS * N_SAMPLES * steps32 / sec32, "unit": "channel-samples/s",
            "ms_per_step": 1e3 * sec32 / steps32, "kernel": engine.last_filter_kernel,
            "roofline_frac": 8.0 * N_CHANS * N_SAMPLES * steps32 / sec32 / 1e9 / hbm_peak,
            "algorithmic_bytes_per_channel_sample": 8, "rel_err_vs_f64_oracle": err32,
        }
        del d_x, d_y
    # ---- cfg3 search shape: 256 channels x 1e5 search samples, dense candidate sweep ------
    # (what find_period(assumed_periods=<8 values>) evaluates per run: 8 x 388 candidates)
    from pyparrm_b200 import _native
    from pyparrm_b200._engine import SearchTile, _vp

    n3, c3 = 100_000, 256
    y3 = torch.randn((n3, c3), dtype=torch.float64, device="cuda", generator=gen).clamp_(-3.0, 3.0)
    ss3 = torch.empty(c3, dtype=torch.float64, device="cuda")
    _native.check(_native.lib.parrm_channel_sumsq(_vp(y3.data_ptr()), _native.F64, c3, c3, n3,
                                                  _vp(ss3.data_ptr()), _vp(stream.cuda_stream)),
                  "parrm_channel_sumsq")
    tile3 = SearchTile(y=y3, sumsq=ss3, indices=torch.arange(n3, dtype=torch.int64, device="cuda"),
                       n_indices=n3, n_chans=c3)
    p3 = 1000 / 145
    grid3 = np.unique(np.concatenate([
        pk * np.concatenate((1 + np.arange(-1e-2, 1e-2 + 1e-4, 1e-4), 1 + np.arange(-1e-3, 1e-3 + 1e-5, 1e-5)))
        for pk in p3 * (1 + 0.03 * np.arange(8))]))
    lo3, hi3 = _sharding.block(len(grid3), world, rank) if world > 1 else (0, len(grid3))
    mine3 = grid3[lo3:hi3]
    engine.evaluate_device(tile3, mine3[:64], 20, 1.0, c3)
    barrier(dist)
    start.record(stream)
    engine.evaluate_device(tile3, mine3, 20, 1.0, c3)
    stop.record(stream)
    barrier(dist)
    sec = max_over_ranks(dist, start.elapsed_time(stop) * 1e-3)
    out["cfg3_search"] = {
        "workload": f"cfg3 search shape: {len(grid3)} candidates (8 assumed periods x the run-1 grid) x "
                    f"{n3} contiguous samples x {c3} channels, bandwidth 20; synthetic tile on the "
                    "device; candidates in contiguous blocks per GPU",
        "value": len(grid3) / sec, "unit": "candidates/s", "seconds": sec, "scaling": "strong",
    }
    del y3, tile3
    # ---- cfg5: candidate sweep, winner only -------------------------------------------
    n_cand, n_fit = 100_000, 100_000
    rng = np.random.default_rng(7)
    t = np.arange(n_fit + 1, dtype=np.float64)
    p_true = FS / FA * (1 + 3e-6)
    y = (np.sin(2 * np.pi * t / p_true) + 0.5 * rng.standard_normal(n_fit + 1))[None, :]
    z = oracle.standardise(y, 3.0)
    tile = engine.tile_from_standardised(z, np.arange(n_fit))
    sweep = (FS / FA) * (1 + np.linspace(-1e-2, 1e-2, n_cand))
    evaluate = lambda blk: engine.evaluate_device(tile, blk, 20, 1.0, 1)  # noqa: E731
    if dist is not None:  # warm-up (workspace allocation, NCCL channel set-up)
        _sharding.minloc_sharded(evaluate, sweep[:2048])
    else:
        evaluate(sweep[:2048])
    barrier(dist)
    t0 = time.perf_counter()
    if dist is not None:
        best, err = _sharding.minloc_sharded(evaluate, sweep)
    else:
        d_err = evaluate(sweep)
        err, best = engine.argmin(d_err)
    torch.cuda.synchronize()
    seconds = max_over_ranks(dist, time.perf_counter() - t0)
    out["cfg5_sweep"] = {
        "workload": f"cfg5: {n_cand} candidate periods x {n_fit} contiguous samples x 1 channel, "
                    "bandwidth 20, lambda 1; candidates in contiguous blocks per GPU, winner by one "
                    "(error, index) pair per rank (_sharding.minloc_sharded)",
        "value": n_cand / seconds, "unit": "candidates/s", "seconds": seconds, "scaling": "strong",
        "winner_rel_err_vs_injected": abs(float(sweep[best]) - p_true) / p_true,
        "winner_error": float(err),
    }
    return out


def bench_search(engine, dist, world, rank, args, dumped):
    """Evaluator throughput on the run-3 shape of the cfg2 recording (candidates sharded over
    ranks by the product's evaluate_sharded), then the whole search through the public API.
    With --dump-outputs the errors of the last timed step go into ``dumped``."""
    import torch

    from pyparrm_b200 import PARRM, _native, _sharding
    from pyparrm_b200.synthetic import make_recording, true_period

    # the search needs the same recording on every rank (SPMD): the 64-channel cfg2 recording
    data = make_recording(N_CHANS, N_SAMPLES, FS, FA, seed=0)
    n_chans, n_samples = data.shape
    rng = np.random.default_rng(0)
    lo, hi = int(np.floor(0.025 * n_samples)), int(n_samples - 2 - np.ceil(0.025 * n_samples))
    indices = np.unique(rng.integers(0, hi - lo, 25000)) + lo       # parrm.py:359-374
    bandwidth = 20
    p0 = FS / FA
    grid = np.unique(p0 * np.concatenate((1 + np.arange(-1e-2, 1e-2 + 1e-4, 1e-4) / 3,
                                          1 + np.arange(-1e-3, 1e-3 + 1e-5, 1e-5) / 3)))
    per_rank = 8 * len(grid)                                          # weak scaling: fixed per GPU
    periods = np.resize(grid, per_rank * world)
    if world > 1:
        (tile,) = _sharding.prepare_tiles_sharded(engine, data, [indices], 3.0)
    else:
        (tile,) = engine.prepare_tiles(data, [indices], 3.0)
    stream = torch.cuda.current_stream()
    steps = args.steps
    evaluate = lambda blk: engine.evaluate_device(tile, blk, bandwidth, 1.0, n_chans)  # noqa: E731

    def one_step():
        if world > 1:  # block per rank + the one all-gather of the errors (SURVEY 8(e))
            return _sharding.evaluate_sharded(evaluate, periods)
        return evaluate(periods).cpu().numpy()

    for _ in range(2):
        one_step()
    barrier(dist)
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record(stream)
    for _ in range(steps):
        errors = one_step()
    stop.record(stream)
    barrier(dist)
    seconds = max_over_ranks(dist, start.elapsed_time(stop) * 1e-3)
    assert errors.shape[0] == per_rank * world and np.isfinite(errors).all()
    if args.dump_outputs and rank == 0:
        dumped["find_period_errors"] = errors

    # FP64 FMA peak of this GPU, measured (no figure for it in MEASURED_PEAKS.json)
    sink = torch.zeros(8, dtype=torch.float64, device="cuda")
    flops = _native.ctypes.c_double(0.0)
    iters = 1 << 15
    for _ in range(2):
        _native.lib.parrm_fp64_fma_burn(iters, sink.data_ptr(), _native.ctypes.byref(flops),
                                        stream.cuda_stream)
    b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    b0.record(stream)
    _native.lib.parrm_fp64_fma_burn(iters, sink.data_ptr(), _native.ctypes.byref(flops),
                                    stream.cuda_stream)
    b1.record(stream)
    torch.cuda.synchronize()
    fp64_peak = flops.value / (b0.elapsed_time(b1) * 1e-3) / 1e12

    m = 2 * bandwidth + 1
    n_idx = len(indices)
    # Flops the device formulation executes per candidate (DESIGN.md 4.4): right-hand sides
    # on the FP64 tensor cores, 2*N*(2bw)*C (the constant row comes from the column sums, once
    # per call); harmonic generator (one complex product = 6 flops + 2 sum adds) 8*N*2bw;
    # sincos + power table ~60*N; solve (2/3)M^3 + 2*C*M^2.
    dmma_flops = 2.0 * n_idx * (2 * bandwidth) * n_chans
    flops_per_cand = dmma_flops + 8.0 * n_idx * 2 * bandwidth + 60.0 * n_idx \
        + (2.0 / 3.0) * m ** 3 + 2.0 * n_chans * m * m
    reference_flops_per_cand = n_idx * (m * (m + 1) + 4.0 * n_chans * m)  # SURVEY 8(d)
    achieved = flops_per_cand * per_rank * steps / seconds / 1e12
    result = {
        "metric": "find_period candidates/sec",
        "value": world * per_rank * steps / seconds, "unit": "candidates/s",
        "ms_per_step": 1e3 * seconds / steps, "steps": steps,
        "config": {"workload": f"evaluator on cfg2 run-3 shape: {n_idx} random samples x {n_chans} "
                               f"channels, bandwidth {bandwidth}, {per_rank} candidates per GPU per step",
                   "sharding": "_sharding.evaluate_sharded: contiguous candidate block per GPU, one "
                               "NCCL all-gather of the errors per step; tiles standardised by channel "
                               "block and all-gathered" if world > 1 else "single GPU"},
        "roofline": {"bound": "fp64", "achieved": achieved, "peak": fp64_peak, "unit": "TFLOP/s",
                     "frac": achieved / fp64_peak, "traffic": None,
                     "dmma_frac": dmma_flops * per_rank * steps / seconds / 1e12 / fp64_peak,
                     "peak_source": "measured here: parrm_fp64_fma_burn (scalar DFMA chains on all "
                                    "SMs; DMMA has the same per-SM flop rate, scripts/micro/dmma_rate.cu)",
                     "flops_per_candidate": flops_per_cand,
                     "reference_flops_per_candidate": reference_flops_per_cand},
    }
    if world == 1:
        # the search's "fp32" mode (PARRM(precision="fp32")): float32 storage of the tile, widened
        # once per call, the fit on the same FP64 tensor path -- same flops, same roofline
        (tile32,) = engine.prepare_tiles(data, [indices], 3.0, "fp32")
        d_per = torch.from_numpy(periods).cuda()
        err64 = engine.evaluate_device(tile, d_per, bandwidth, 1.0, n_chans)
        for _ in range(2):
            err32 = engine.evaluate_device(tile32, d_per, bandwidth, 1.0, n_chans)
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record(stream)
        for _ in range(steps):
            err32 = engine.evaluate_device(tile32, d_per, bandwidth, 1.0, n_chans)
        f1.record(stream)
        torch.cuda.synchronize()
        sec32 = f0.elapsed_time(f1) * 1e-3
        result["fp32_mode"] = {
            "what": "same candidates on the float32 tile of PARRM(precision='fp32'): float32 storage, "
                    "widened once per call, fit on the FP64 tensor path (no FP32-pipe kernel: "
                    "DESIGN.md 4.4)",
            "value": per_rank * steps / sec32, "unit": "candidates/s",
            "roofline_frac_of_fp64_peak": flops_per_cand * per_rank * steps / sec32 / 1e12 / fp64_peak,
            "max_rel_err_vs_fp64_tile": float(((err32 - err64).abs() / err64.abs()).max().item()),
            "tolerance": 1e-4,
        }
        del tile32
    # the whole search through the public API (host array in, period out): three coarse-to-fine
    # grid runs + lock-step Nelder-Mead, ~1 800 objective evaluations (SURVEY 3.2); under
    # enable_sharding() every rank uploads only its channel block and evaluates its candidates
    searcher = PARRM(data, FS, FA, verbose=False)
    searcher.find_period(random_seed=0)  # first call builds tiles' workspace; timed call below
    barrier(dist)
    launches0 = engine.launches
    t0 = time.perf_counter()
    searcher.find_period(random_seed=0)
    api_seconds = max_over_ranks(dist, time.perf_counter() - t0)
    result["public_api"] = {
        "call": "PARRM(data, 2000, 130).find_period(random_seed=0) on the 64 x 1.2M recording"
                + (" under enable_sharding()" if world > 1 else ""),
        "seconds": api_seconds, "gpu_launches": engine.launches - launches0,
        "period": float(searcher.period),
        "rel_err_vs_injected_period": abs(float(searcher.period) - true_period(FS, FA))
        / true_period(FS, FA),
    }
    if rank == 0 and world == 1:
        result["cpu_baseline"] = cpu_search_baseline(data, indices, grid, bandwidth)
    return result


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50,
                    help="timed passes of the headline, e2e, e2e_variants and find_period legs "
                         "(the strong-scaling, standardise and power-capped figures time fixed "
                         "counts of their own)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (--impl b200)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    if args.dump_outputs:  # an unwritable DIR fails here, not after the whole run
        os.makedirs(args.dump_outputs, exist_ok=True)
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()

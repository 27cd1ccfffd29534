"""Re-calibrating an open stream (filter_stream(history=...), recent(), set_filter()): what it
costs.

1. Per-push wall time, p50 / p99, with history=0 against history = 10 s, for 384 channels of
   int16 in / float32 out at a cfg4-like period (30 kHz / 130 Hz, "future" taps, half-width
   2311), blocks of 30 / 300 / 3000 samples (the setup of scripts/stream_latency.py).
2. Wall time of one re-calibration -- recent(window) + PARRM(window) + find_period() +
   create_filter() + set_filter(), ended by a device synchronise -- for 1 s and 10 s windows at
   30 kHz x 384 channels and a 10 s window at 2 kHz x 64 channels (best and median of --recals).
3. Per-push wall time (300- and 3000-sample blocks) while another host thread re-calibrates the
   same stream over and over, next to the same pushes with no re-calibration running.

Usage: python scripts/recalibrate_latency.py [--out FILE] [--pushes 500] [--warmup 50]
"""

from __future__ import annotations

import argparse
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import parrm_oracle as oracle  # noqa: E402
from pyparrm_b200 import PARRM, _engine  # noqa: E402
from pyparrm_b200._stream import FilterStream  # noqa: E402
from pyparrm_b200.synthetic import make_recording  # noqa: E402
from scripts.stream_latency import gpu_identity  # noqa: E402

FS4, FA = 30000, 130
PER4 = FS4 / FA * (1 + 3e-6)


def int16_blocks(n_chans, n, count=32, seed=0):
    rec = make_recording(n_chans, n * count, FS4, FA, seed=seed) * 300
    return [np.ascontiguousarray(rec[:, i * n:(i + 1) * n]).astype(np.int16) for i in range(count)]


def push_times(stream, blocks, pushes, warmup, stop=None):
    times = np.empty(pushes)
    for i in range(warmup + pushes):
        t0 = time.perf_counter()
        stream.push(blocks[i % len(blocks)])
        t1 = time.perf_counter()
        if i >= warmup:
            times[i - warmup] = t1 - t0
    if stop is not None:
        stop.set()
    us = times * 1e6
    return np.percentile(us, 50), np.percentile(us, 99)


def recalibrate(stream, window, fs, hw):
    """One re-calibration from the stream's own recent samples; returns its wall time."""
    import torch

    torch.cuda.synchronize()
    t0 = time.perf_counter()
    cal = PARRM(stream.recent(window), fs, FA, verbose=False)
    cal.find_period(random_seed=0)
    cal.create_filter(filter_half_width=hw, filter_direction="future")
    stream.set_filter(cal)
    torch.cuda.synchronize()
    return time.perf_counter() - t0, cal.period


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--pushes", type=int, default=500)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--recals", type=int, default=5)
    args = ap.parse_args()
    engine = _engine.get_engine()
    taps = oracle.tap_offsets(PER4, PER4 / 50, 2311, 0, "future")
    lines = [f"# scripts/recalibrate_latency.py on {gpu_identity()} (name, power limit, max SM clock)",
             "# 1. per-push wall time, push() call -> returned NumPy array; 384 ch int16 in, "
             "float32 out, 'future' taps",
             f"#    cfg4-like period 30000/130 samples, half-width 2311 ({len(taps)} taps); "
             f"{args.pushes} timed pushes after {args.warmup}",
             "block  history   p50_us   p99_us"]
    for n in (30, 300, 3000):
        blocks = int16_blocks(384, n)
        for history in (0, 10 * FS4):
            stream = FilterStream(engine, taps, out_dtype=np.float32, history=history)
            p50, p99 = push_times(stream, blocks, args.pushes, args.warmup)
            stream.close()
            lines.append(f"{n:5d}  {history:7d}  {p50:7.1f}  {p99:7.1f}")
            print(lines[-1], flush=True)

    lines += ["", "# 2. one re-calibration: recent(window) + PARRM + find_period + create_filter"
              " + set_filter, to a device synchronise",
              f"#    best / median of {args.recals}; half-width 2311 at 30 kHz, 2000 at 2 kHz",
              "fs_hz  channels  window_s   best_ms  median_ms  period"]
    for fs, n_chans, seconds in ((FS4, 384, 1), (FS4, 384, 10), (2000, 64, 10)):
        window = seconds * fs
        hw = 2311 if fs == FS4 else 2000
        per = fs / FA * (1 + 3e-6)
        rec = (make_recording(n_chans, window, fs, FA, seed=1) * 300).astype(np.int16)
        stream = FilterStream(engine, oracle.tap_offsets(per, per / 50, hw, 0, "future"),
                              out_dtype=np.float32, history=window)
        for t in range(0, window, fs // 10):
            stream.push(rec[:, t:t + fs // 10])
        recalibrate(stream, window, fs, hw)  # warm-up: kernels load, workspaces grow
        runs = [recalibrate(stream, window, fs, hw) for _ in range(args.recals)]
        dts = np.array([r[0] for r in runs]) * 1e3
        lines.append(f"{fs:5d}  {n_chans:8d}  {seconds:8d}  {dts.min():8.1f}  {np.median(dts):9.1f}"
                     f"  {runs[-1][1]:.6f}")
        print(lines[-1], flush=True)
        stream.close()

    lines += ["", "# 3. per-push wall time with another host thread re-calibrating the same stream"
              " (1 s window, 384 ch at 30 kHz) back to back",
              "block  recalibrating   p50_us   p99_us  recals_during"]
    window = FS4
    for n in (300, 3000):
        blocks = int16_blocks(384, n)
        for busy in (False, True):
            stream = FilterStream(engine, taps, out_dtype=np.float32, history=window)
            for _ in range(-(-window // n)):
                stream.push(blocks[0])
            stop, count = threading.Event(), [0]

            def worker():
                while not stop.is_set():
                    recalibrate(stream, window, FS4, 2311)
                    count[0] += 1

            th = threading.Thread(target=worker) if busy else None
            if th is not None:
                th.start()
                time.sleep(0.2)  # the first re-calibration is under way
            p50, p99 = push_times(stream, blocks, args.pushes, args.warmup, stop)
            if th is not None:
                th.join()
            stream.close()
            lines.append(f"{n:5d}  {'yes' if busy else 'no':13s}  {p50:7.1f}  {p99:7.1f}  "
                         f"{count[0]}")
            print(lines[-1], flush=True)

    text = "\n".join(lines) + "\n"
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()

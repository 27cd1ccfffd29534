"""Streaming filter (PARRM.filter_stream): per-push latency and streamed throughput.

1. Per-push wall time, from the push() call to the returned NumPy array, p50 / p99 over
   --pushes pushes (after --warmup), for 384 channels of int16 at a cfg4-like period
   (30 kHz / 130 Hz, half-width 2311) with "future" (latency 0) and "both" taps, blocks of
   30 / 300 / 3000 samples, eager launches vs CUDA-graph replays, float32 results.  The p50 of
   the first and the last 100 timed pushes is printed too: per-push time must follow the block
   size, not how much has been pushed.
2. Aggregate channel-samples/s of streaming cfg2's recording (64 x 1.2 M float64 at 2 kHz,
   160 taps) in 1 s blocks, next to filter_data() on the whole array (best of 3, warm).

Usage: python scripts/stream_latency.py [--out FILE] [--pushes 1000] [--warmup 50]
"""

from __future__ import annotations

import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import parrm_oracle as oracle  # noqa: E402
from pyparrm_b200 import _engine  # noqa: E402
from pyparrm_b200._stream import FilterStream  # noqa: E402
from pyparrm_b200.synthetic import make_recording  # noqa: E402


def gpu_identity() -> str:
    try:
        return subprocess.run(
            ["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
            capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.SubprocessError):
        return "unknown (nvidia-smi not available)"


def push_latency(engine, taps, n, graphs, pushes, warmup, n_chans=384):
    rng = np.random.default_rng(n)
    blocks = [rng.integers(-3000, 3000, (n_chans, n)).astype(np.int16) for _ in range(32)]
    stream = FilterStream(engine, taps, out_dtype=np.float32, graphs=graphs)
    times = np.empty(pushes)
    for i in range(warmup + pushes):
        block = blocks[i % len(blocks)]
        t0 = time.perf_counter()
        y = stream.push(block)
        t1 = time.perf_counter()
        if i >= warmup:
            times[i - warmup] = t1 - t0
    assert y.dtype == np.float32 and y.shape == (n_chans, n)
    stream.close()
    us = times * 1e6
    return (np.percentile(us, 50), np.percentile(us, 99), np.median(us[:100]),
            np.median(us[-100:]), stream.n_pushed)


def aggregate(engine, reps=3):
    fs, fa, n = 2000, 130, 1_200_000
    x = make_recording(64, n, fs, fa, seed=0)
    per = fs / fa * (1 + 3e-6)
    taps = oracle.tap_offsets(per, per / 50, 2000, 0, "both")
    rows = []
    whole = engine.filter_host(x, taps)  # warm-up: plans, the specialised kernel's build
    best_whole = None
    for _ in range(reps):
        t0 = time.perf_counter()
        engine.filter_host(x, taps)
        dt = time.perf_counter() - t0
        best_whole = dt if best_whole is None else min(best_whole, dt)
    blocks = [np.ascontiguousarray(x[:, t:t + fs]) for t in range(0, n, fs)]
    for graphs in (False, True):
        best = None
        for _ in range(reps):
            stream = FilterStream(engine, taps, graphs=graphs)
            outs = []
            t0 = time.perf_counter()
            for b in blocks:
                outs.append(stream.push(b))
            outs.append(stream.close())
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
        got = np.concatenate(outs, axis=1)
        err = float(np.abs(got - whole).max() / np.abs(x).max())
        rows.append((graphs, best, err))
    return x.size, best_whole, rows, len(taps)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--pushes", type=int, default=1000)
    ap.add_argument("--warmup", type=int, default=50)
    args = ap.parse_args()
    engine = _engine.get_engine()
    lines = [f"# scripts/stream_latency.py on {gpu_identity()} (name, power limit, max SM clock)",
             "# per-push wall time, push() call -> returned NumPy array; 384 ch int16 in, float32 out",
             "# cfg4-like period 30000/130 samples, half-width 2311; "
             f"{args.pushes} timed pushes after {args.warmup} warm-up pushes",
             "direction  taps  latency  block  mode   p50_us   p99_us  p50_first100  p50_last100  pushed"]
    per = 30000 / 130 * (1 + 3e-6)
    for direction in ("future", "both"):
        taps = oracle.tap_offsets(per, per / 50, 2311, 0, direction)
        for n in (30, 300, 3000):
            for graphs in (False, True):
                p50, p99, first, last, pushed = push_latency(engine, taps, n, graphs, args.pushes,
                                                             args.warmup)
                lines.append(f"{direction:9s}  {len(taps):4d}  {max(0, -int(taps[0])):7d}  {n:5d}  "
                             f"{'graph' if graphs else 'eager':5s}  {p50:7.1f}  {p99:7.1f}  "
                             f"{first:12.1f}  {last:11.1f}  {pushed}")
                print(lines[-1], flush=True)
    size, t_whole, rows, n_taps = aggregate(engine)
    lines.append("")
    lines.append(f"# cfg2 recording 64 x 1 200 000 float64, {n_taps} taps (both), float64 out; best of 3")
    lines.append(f"filter_data whole array      {t_whole * 1e3:9.1f} ms  {size / t_whole / 1e9:7.3f} G ch-samples/s")
    for graphs, dt, err in rows:
        lines.append(f"stream, 1 s blocks, {'graph' if graphs else 'eager'}    {dt * 1e3:9.1f} ms  "
                     f"{size / dt / 1e9:7.3f} G ch-samples/s  (max |stream - whole| / max |x| = {err:.1e})")
    text = "\n".join(lines) + "\n"
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text)


if __name__ == "__main__":
    main()

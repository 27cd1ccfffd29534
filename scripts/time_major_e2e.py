#!/usr/bin/env python
"""Time-major ("interleaved", [times, channels]) recordings end to end on one GPU.

Records, with the card's name and power limit read in the same run:
  1. parrm_transpose's rate (bytes read + written over kernel time, CUDA events) for the type
     pairs the pipelines use, against the 6.55 TB/s HBM copy rate measured on a B200;
  2. cfg2 (64 x 1.2 M float64) through filter_data: time-major view against the C-order array;
  3. a cfg4 48-channel share and the full 384 x 9 M cfg4, int16 in, float32 out:
       (a) np.ascontiguousarray(mm.T) + filter_data + a transpose back into a [T, C] array,
       (b) filter_data(mm.T, out=out.T) straight into a [T, C] array,
     with the recording and the result pageable, then page-locked;
  4. find_period on a time-major cfg2-shaped recording against np.ascontiguousarray + find_period.
Outputs of each pair are compared at the timed size.

python scripts/time_major_e2e.py [--out PATH] [--skip-full]
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pyparrm_b200 import PARRM, _engine, _native  # noqa: E402
from pyparrm_b200._engine import pin_array  # noqa: E402
from pyparrm_b200.synthetic import make_recording  # noqa: E402

HBM_COPY_TBS = 6.55
lines = []


def say(text=""):
    print(text, flush=True)
    lines.append(text)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "nvidia-smi unavailable"


def timed(fn, reps=1, warm=True):
    if warm:
        fn()
    best = float("inf")
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        best = min(best, time.perf_counter() - t0)
    return best


def transpose_rates():
    import torch

    say("1. parrm_transpose, [rows, cols] -> [cols, rows], 20 launches timed with CUDA events")
    rows, cols = 2_000_000, 384
    es = {_native.F64: 8, _native.F32: 4, _native.I16: 2}
    for s, d, name in ((_native.I16, _native.F32, "int16 -> float32"),
                       (_native.I16, _native.F64, "int16 -> float64"),
                       (_native.F32, _native.F32, "float32 -> float32"),
                       (_native.F64, _native.F32, "float64 -> float32"),
                       (_native.F64, _native.F64, "float64 -> float64")):
        src = torch.empty(rows * cols * es[s], dtype=torch.uint8, device="cuda")
        dst = torch.empty(rows * cols * es[d], dtype=torch.uint8, device="cuda")
        sp = torch.cuda.current_stream().cuda_stream

        def run():
            _native.check(_native.lib.parrm_transpose(src.data_ptr(), s, rows, cols, cols,
                                                      dst.data_ptr(), d, rows, sp), "transpose")

        for _ in range(3):
            run()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(20):
            run()
        b.record()
        b.synchronize()
        sec = a.elapsed_time(b) / 1e3 / 20
        gbs = rows * cols * (es[s] + es[d]) / sec / 1e9
        say(f"   {name:20s} {rows} x {cols}: {sec * 1e3:7.3f} ms, {gbs:7.0f} GB/s "
            f"({gbs / 1e3 / HBM_COPY_TBS:.0%} of the {HBM_COPY_TBS} TB/s HBM copy rate)")


def cfg2_filter():
    say("\n2. cfg2 filter_data, 64 x 1.2 M float64, half-width 2000, both directions")
    x = make_recording(64, 1_200_000, 2000, 130, seed=0)
    base = np.ascontiguousarray(x.T)
    tm = base.T
    parrm = PARRM(x, 2000, 130, verbose=False)
    parrm._period = np.float64(2000 / 130 * (1 + 3e-6))
    parrm.create_filter(filter_half_width=2000, filter_direction="both")
    res = {}
    for name, data in (("C-order", x), ("time-major", tm)):
        sec = timed(lambda: res.__setitem__(name, parrm.filter_data(data)), reps=5)
        say(f"   {name:10s} {sec * 1e3:8.1f} ms  ({64 * 1.2e6 / sec / 1e9:.2f} G channel-samples/s)")
    diff = np.abs(res["C-order"] - res["time-major"]).max() / np.abs(x).max()
    say(f"   max |time-major - C-order| = {diff:.2e} of the input scale")


def cfg4(n_chans, reps, warm=True):
    n, fs, fa = 9_000_000, 30000, 130
    say(f"\n3. cfg4 {n_chans} ch x {n} samples, int16 [T, C] in, float32 [T, C] out, one-sided "
        "default-width filter")
    rng = np.random.default_rng(0)
    period = fs / fa * (1 + 3e-6)
    mm = np.empty((n, n_chans), dtype=np.int16)       # what np.load(path, mmap_mode="r") maps
    for t0 in range(0, n, 1 << 20):                   # frames in blocks: artefact + noise
        t = np.arange(t0, min(t0 + (1 << 20), n))
        wave = 600 * sum(np.sin(2 * np.pi * k * t / period + k) / k for k in range(1, 6))
        noise = 200 * rng.standard_normal((t.size, n_chans), dtype=np.float32)
        mm[t0:t0 + t.size] = np.clip(np.round(noise + wave[:, None]), -32768, 32767)
    parrm = PARRM(mm.T, fs, fa, verbose=False)
    parrm._period = np.float64(period)
    parrm.create_filter(filter_direction="past")
    res_a = np.empty((n, n_chans), dtype=np.float32)
    res_b = np.empty((n, n_chans), dtype=np.float32)

    def way_a():
        x = np.ascontiguousarray(mm.T)
        y = parrm.filter_data(x, out_dtype=np.float32)
        res_a[...] = y.T

    def way_b():
        parrm.filter_data(mm.T, out=res_b.T)

    c_only = {}

    def c_order_filter(x):
        c_only["t"] = timed(lambda: parrm.filter_data(x, out_dtype=np.float32), reps, warm)

    for label in ("pageable", "pinned"):
        handles = [pin_array(mm), pin_array(res_a), pin_array(res_b)] if label == "pinned" else []
        try:
            ta = timed(way_a, reps, warm)
            tb = timed(way_b, reps, warm)
            xc = np.ascontiguousarray(mm.T)
            hc = [pin_array(xc)] if label == "pinned" else []
            c_order_filter(xc)
            for h in hc:
                h.release()
            del xc
        finally:
            for h in handles:
                h.release()
        gb = mm.nbytes / 1e9 + res_b.nbytes / 1e9
        diff = max(float(np.abs(res_a[i:i + (1 << 20)] - res_b[i:i + (1 << 20)]).max())
                   for i in range(0, n, 1 << 20)) / float(np.abs(mm).max())
        say(f"   {label:8s} (a) host transpose + filter_data + transpose back: {ta:7.3f} s")
        say(f"   {label:8s} (b) filter_data(mm.T, out=out.T):                    {tb:7.3f} s "
            f"({gb / tb:5.1f} GB/s of int16 in + float32 out)")
        say(f"   {label:8s}     filter_data on the C-order copy (same bytes):      "
            f"{c_only['t']:7.3f} s -> (b) / C-order = {tb / c_only['t']:.2f}")
        say(f"   {label:8s}     max |(a) - (b)| = {diff:.2e} of the input scale; kernel "
            f"{_engine.get_engine().last_filter_kernel}")


def search():
    say("\n4. find_period, cfg2-shaped 64 x 1.2 M float64 time-major recording")
    x = make_recording(64, 1_200_000, 2000, 130, seed=1)
    tm = np.ascontiguousarray(x.T).T
    del x
    out = {}

    def host_path():
        p = PARRM(np.ascontiguousarray(tm), 2000, 130, verbose=False)
        p.find_period(random_seed=0)
        out["host"] = p.period

    def device_path():
        p = PARRM(tm, 2000, 130, verbose=False)
        p.find_period(random_seed=0)
        out["tm"] = p.period

    th = timed(host_path, 3)
    td = timed(device_path, 3)
    say(f"   np.ascontiguousarray + find_period: {th:7.3f} s")
    say(f"   find_period(time-major view):       {td:7.3f} s")
    say(f"   periods equal bit for bit: {out['host'] == out['tm']} ({out['tm']!r})")


def narrow_subsets():
    """Channel subsets of a 385-channel int16 file read as rows of the file (the upload carries
    all 385 channels) against the host copy of the channels asked for: where the width rule
    (``_engine._TIME_MAJOR_MAX_WIDTH``) should sit."""
    n, n_file, fs, fa = 9_000_000, 385, 30000, 130
    say(f"\n5. channel subsets of an int16 [{n}, {n_file}] file, float32 out (pageable): rows of the "
        "file through the device transpose vs the host copy of the subset")
    rng = np.random.default_rng(3)
    mm = np.empty((n, n_file), dtype=np.int16)
    for t0 in range(0, n, 1 << 20):
        t1 = min(t0 + (1 << 20), n)
        mm[t0:t1] = rng.integers(-2000, 2000, (t1 - t0, n_file), dtype=np.int16)
    parrm = PARRM(mm[:, :1].T, fs, fa, verbose=False)
    parrm._period = np.float64(fs / fa * (1 + 3e-6))
    parrm.create_filter(filter_direction="past")
    width = _engine._TIME_MAJOR_MAX_WIDTH
    for n_chans in (1, 8, 24, 48):
        view = mm[:, n_file - n_chans:].T
        got = {}
        for name, limit in (("rows", n_file), ("host copy", 0)):
            _engine._TIME_MAJOR_MAX_WIDTH = limit
            sec = timed(lambda: got.__setitem__(name, parrm.filter_data(view, out_dtype=np.float32)),
                        2)
            got[name + " s"] = sec
        _engine._TIME_MAJOR_MAX_WIDTH = width
        diff = float(np.abs(got["rows"] - got["host copy"]).max()) / 2000
        say(f"   C = {n_chans:3d} (rows {n_file / n_chans:5.1f}x wider): rows {got['rows s']:6.3f} s, "
            f"host copy {got['host copy s']:6.3f} s, max diff {diff:.1e} of the scale; rule picks "
            f"{'rows' if n_file <= width * n_chans else 'host copy'}")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("profiles", "r3", "time_major.txt"))
    ap.add_argument("--skip-full", action="store_true", help="leave out the 384-channel cfg4")
    args = ap.parse_args()
    say("Time-major recordings end to end (scripts/time_major_e2e.py)")
    say(f"GPU: {card()}")
    transpose_rates()
    cfg2_filter()
    cfg4(48, 3)
    if not args.skip_full:
        cfg4(384, 1, warm=False)   # plan, kernel and ring already warm from the share
    search()
    narrow_subsets()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()

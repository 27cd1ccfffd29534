"""SHA-256 digests of the gather filter's outputs on fixed seeded cases, one line per case:
the whole-recording gather kernels (forced with KERNEL_GATHER, float64 and float32), the
batched sweep, and two stream sessions that switch taps.  Every input carries NaN and +-Inf
samples.  Two builds that print the same lines computed the same bytes.

    python scripts/gather_digests.py [repo root to import pyparrm_b200 from]   (needs a GPU)
"""
import hashlib
import os
import sys

ROOT = os.path.abspath(sys.argv[1]) if len(sys.argv) > 1 else os.path.dirname(
    os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from oracle.parrm_oracle import tap_offsets  # noqa: E402
from pyparrm_b200 import PARRM, _engine, _native  # noqa: E402
from pyparrm_b200._stream import FilterStream  # noqa: E402


def recording(seed, n_chans, n):
    x = np.random.default_rng(seed).standard_normal((n_chans, n)) * 50
    x[0, n // 3] = np.nan
    x[-1, n // 2] = np.inf
    x[-1, n // 2 + 7] = -np.inf
    return x


def digest(name, y, kernel=""):
    y = y.cpu().numpy() if hasattr(y, "is_cuda") else y
    h = hashlib.sha256(np.ascontiguousarray(y).tobytes()).hexdigest()
    print(f"{name:34s} {kernel:28s} {y.dtype} {y.shape} {h}", flush=True)


class Taps:  # what FilterStream.set_filter reads of a PARRM object
    def __init__(self, taps):
        self._taps, self._filter = np.asarray(taps, dtype=np.int32), np.zeros(1)

    def _tap_offsets(self):
        return self._taps


def stream_session(engine, x, taps_list, sizes, switch_at, **kw):
    stream, outs, t = FilterStream(engine, taps_list[0], **kw), [], 0
    for i, n in enumerate(sizes):
        if i == switch_at:
            stream.set_filter(Taps(taps_list[1]))
        outs.append(stream.push(x[:, t:t + n]))
        t += n
    outs.append(stream.close())
    return torch.cat(outs, dim=1) if hasattr(outs[0], "is_cuda") else np.concatenate(outs, axis=1)


def main():
    engine = _engine.get_engine()
    p = 30000 / 130 * (1 + 3e-6)
    cases = [("interior 16x400000", recording(1, 16, 400_000), tap_offsets(p, p / 50, 2311, 0, "both")),
             ("ragged 3x1777", recording(2, 3, 1_777), tap_offsets(15.38, 0.3, 500, 3, "past")),
             ("global 2x90000", recording(3, 2, 90_000), tap_offsets(230.77, 4.6, 40_000, 0, "both"))]
    for name, x, taps in cases:
        for dt in (torch.float64, torch.float32):
            y = engine.filter_device(torch.from_numpy(x).cuda().to(dt), taps,
                                     kernel=_native.KERNEL_GATHER)
            digest(f"apply {name} {str(dt)[6:]}", y, engine.last_filter_kernel)

    x = recording(4, 2, 9_000)
    parrm = PARRM(x, 2000, 130, verbose=False)
    parrm._period = np.float64(2000 / 130 * (1 + 3e-6))
    out, _ = parrm.filter_sweep([dict(filter_half_width=2000), dict(),
                                 dict(filter_direction="past", omit_n_samples=5),
                                 dict(filter_half_width=700, filter_direction="future")])
    digest("filter_sweep 2x9000 x4 sets", out, engine.last_filter_kernel)

    x = recording(5, 4, 200_000)
    sizes = [1, 30_011, 65_536, 7, 41_000, 63_445]
    narrow, wide = tap_offsets(229.9, 4.6, 2_000, 0, "past"), tap_offsets(230.77, 4.6, 40_000, 0, "both")
    digest("stream numpy fp64 narrow->wide", stream_session(engine, x, [narrow, wide], sizes, 3,
                                                             history=82_000))
    x = recording(6, 6, 60_000)
    sizes = [13, 300, 3000, 997, 5000, 301, 1] * 6
    sizes.append(x.shape[1] - sum(sizes))
    taps_list = [tap_offsets(p, p / 50, 2311, 0, "future"), tap_offsets(30000 / 131, p / 50, 1500, 0, "both")]
    for prec in ("fp64", "fp32"):
        digest(f"stream cuda {prec} future->both", stream_session(
            engine, torch.from_numpy(x).cuda(), taps_list, sizes, 9, history=6_000,
            max_chunk=4096, precision=prec))


if __name__ == "__main__":
    main()

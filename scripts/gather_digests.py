"""SHA-256 digests of the gather filter's outputs on fixed seeded cases, one line per case:
the whole-recording gather kernels (forced with KERNEL_GATHER, float64 and float32), the
batched sweep, and two stream sessions that switch taps.  Every input carries NaN and +-Inf
samples.  Then the engine's host pipelines, each line with the launches it enqueued: the
filter's ring at a small chunk size (pageable and pinned float64, int16 and time-major input,
C-ordered and time-major ``out=``, float32 compute and output), time shards, and the period
search's tiles (``y``, ``sumsq``) of host, pinned, time-major and CUDA-tensor recordings.  Two
builds that print the same lines computed the same bytes.

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


def counted(engine, name, fn):
    """Digest of what ``fn()`` returns (an array or a list of tiles) and the launches it made."""
    launches = engine.launches
    got = fn()
    if isinstance(got, list):  # search tiles: y and sumsq of every tile
        got = np.concatenate([np.concatenate([t.y.double().cpu().numpy().ravel(),
                                              t.sumsq.cpu().numpy()]) for t in got])
    digest(name, got, f"launches {engine.launches - launches}")


def host_pipelines(engine):
    taps = tap_offsets(15.38, 0.3, 100, 3, "both")
    x = recording(7, 40, 3_000)                                    # several rows per chunk
    long_x = recording(8, 3, 60_000)                               # windows of one row
    i16 = (np.random.default_rng(9).standard_normal((5, 70_000)) * 900).astype(np.int16)
    wide = (np.random.default_rng(10).standard_normal((200_000, 12)) * 900).astype(np.int16)
    tm64 = recording(11, 7, 200_000).T.copy()
    _engine._CHUNK_BYTES = 1 << 16                                 # many slots, many reuses
    # (name, C-contiguous array, the recording as a view of it, filter_host keywords)
    cases = [("x", x, None, {}), ("long", long_x, None, {}), ("i16", i16, None, {}),
             ("tm i16 ld 12", wide, lambda b: b[:, 2:9].T, {}),
             ("tm f64 ld 7", tm64, lambda b: b.T, {}),
             ("x fp32", x, None, dict(precision="fp32")),
             ("i16 f32 out", i16, None, dict(out_dtype=np.float32)),
             ("tm fp32 f32 out", wide, lambda b: b[:, 2:9].T,
              dict(precision="fp32", out_dtype=np.float32))]
    for name, base, view, kw in cases:
        for pinned in (False, True):
            if pinned:
                base = base.copy()
                handle = _engine.pin_array(base)
            data = base if view is None else view(base)
            tag = f"filter_host {name}{' pinned' if pinned else ''}"
            counted(engine, tag, lambda: engine.filter_host(data, taps, **kw))
            (n_chans, n), dt = data.shape, kw.get("out_dtype", np.float64)
            for out_name, out in (("C out", np.full((n_chans, n), 7.0, dt)),
                                  ("tm out", np.full((n, n_chans + 3), 7.0, dt)[:, 2:-1].T)):
                counted(engine, f"{tag} {out_name}",
                        lambda: engine.filter_host(data, taps, out=out, **kw))
            if pinned:
                handle.release()
    for prec in ("fp64", "fp32"):
        x0, t0, t1, n = 20_000, 21_000, 41_000, long_x.shape[1]
        counted(engine, f"filter_shard {prec}", lambda: engine.filter_shard(
            long_x[:, x0:t1 + 200], taps, x0, t0, t1, n, prec))

    rng = np.random.default_rng(12)
    rec = np.random.default_rng(13).standard_normal((23, 40_001)) * 50
    rec[3, 1000:1010] = 900.0                                      # outliers
    idx_sets = [np.sort(rng.choice(rec.shape[1] - 1, m, replace=False)) for m in (3_000, 777)]
    tm_rec = rec.T.copy().T                                        # time-major, ld 23
    pinned = rec.copy()
    handle = _engine.pin_array(pinned)
    for chunk in (5 * rec.shape[1] * 8, 23 * 8 * 997):             # 5 rows; 1 row, 997 samples
        _engine._SEARCH_CHUNK_BYTES = chunk
        for prec in ("fp64", "fp32"):
            for name, data, share in (("host", rec, 0.5), ("pinned", pinned, 0.5),
                                      ("time-major", tm_rec, 0.5), ("time-major host", tm_rec, 0.0),
                                      ("cuda", torch.from_numpy(rec).cuda(), 0.5)):
                _engine._SEARCH_DEVICE_SHARE = share
                counted(engine, f"prepare_tiles {name} {prec} {chunk}",
                        lambda: engine.prepare_tiles(data, idx_sets, 3.0, prec))
    handle.release()


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
    host_pipelines(engine)


if __name__ == "__main__":
    main()

"""Device engine: what ``pyparrm_b200.PARRM`` calls for every piece of arithmetic.

One engine per process and GPU.  PyTorch owns device memory, pinned staging buffers and
streams; all computation goes through the C ABI in ``_native`` (hand-written sm_100a
kernels).  There is no CPU path: constructing the engine without a CUDA device raises.

Host <-> device traffic uses a three-slot ring on three streams (H2D, compute, D2H), so the
NumPy-in / NumPy-out API of the reference (``parrm.py:120-121``, ``:866-875``) overlaps copies
with the kernels.  Pinned host arrays (see :func:`pinned_empty`) are copied directly; pageable
ones are staged through pinned buffers with a threaded memcpy.
"""

from __future__ import annotations

import ctypes
import os
import threading
from dataclasses import dataclass, field

import numpy as np

from . import _native
from ._native import check, lib

_CHUNK_BYTES = int(os.environ.get("PYPARRM_B200_CHUNK_MB", "32")) << 20
# the search prologue reads every row once and writes next to nothing back: bigger chunks,
# fewer launches (five kernels per chunk), the copy/compute overlap is the same
_SEARCH_CHUNK_BYTES = int(os.environ.get("PYPARRM_B200_SEARCH_CHUNK_MB", "128")) << 20
_PINNED_OUT_LIMIT = int(os.environ.get("PYPARRM_B200_PINNED_OUT_MB", "2048")) << 20
_EVAL_WS_LIMIT = int(os.environ.get("PYPARRM_B200_EVAL_WS_MB", "1024")) << 20
_N_SLOTS = 3
_COPY_THREADS = max(1, min(int(os.environ.get("PYPARRM_B200_COPY_THREADS", "8")), (os.cpu_count() or 1)))


def _vp(ptr: int) -> ctypes.c_void_p:
    return ctypes.c_void_p(int(ptr))


def _threaded_memmove(dst: int, src: int, nbytes: int) -> None:
    """Host-to-host copy between a pageable array and a pinned staging buffer, on the
    library's copy threads (``parrm_host_copy``; the call releases the GIL)."""
    check(lib.parrm_host_copy(_vp(dst), _vp(src), nbytes, _COPY_THREADS), "parrm_host_copy")


def pinned_empty(shape, dtype=np.float64) -> np.ndarray:
    """Uninitialised page-locked NumPy array (fast, asynchronous host<->device copies)."""
    import torch

    tdtype = {np.dtype(np.float64): torch.float64, np.dtype(np.float32): torch.float32}[
        np.dtype(dtype)
    ]
    return torch.empty(tuple(shape), dtype=tdtype, pin_memory=True).numpy()


def is_pinned(array: np.ndarray) -> bool:
    return bool(lib.parrm_host_is_pinned(_vp(array.ctypes.data)))


class pin_array:
    """Page-lock an existing C-contiguous NumPy array in place (``cudaHostRegister``), so that
    every later ``find_period`` / ``filter_data`` on it copies straight from the caller's
    memory instead of staging each call through pinned buffers.  Worth it when the same
    recording is used more than once (registering costs about as much as one staged pass).

    ``handle = pin_array(data)`` ... ``handle.release()``; also a context manager.  The array
    must stay alive and must not be resized while registered."""

    def __init__(self, array: np.ndarray):
        if not isinstance(array, np.ndarray) or not array.flags.c_contiguous:
            raise TypeError("pin_array needs a C-contiguous NumPy array")
        self.array = array
        self._ptr = None
        if array.nbytes and not is_pinned(array):
            check(lib.parrm_host_register(_vp(array.ctypes.data), array.nbytes),
                  "parrm_host_register")
            self._ptr = array.ctypes.data

    def release(self) -> None:
        if self._ptr is not None:
            check(lib.parrm_host_unregister(_vp(self._ptr)), "parrm_host_unregister")
            self._ptr = None

    def __enter__(self):
        return self.array

    def __exit__(self, *exc) -> None:
        self.release()


@dataclass
class SearchTile:
    """Standardised samples of one search run, resident on the device."""

    y: object          # torch [n_indices, n_chans] float64 (float32 in the fp32 mode), sample-major
    sumsq: object      # torch [n_chans] float64
    indices: object    # torch [n_indices] int64
    n_indices: int
    n_chans: int

    @property
    def y_code(self) -> int:
        import torch

        return _native.F32 if self.y.dtype == torch.float32 else _native.F64


@dataclass(eq=False)
class _StreamState:
    """Device state of one streaming filter (``DeviceEngine.stream_open``)."""

    taps: np.ndarray
    d_taps: object
    max_chunk: int
    code: int           # compute type of the ring and the kernel
    latency: int
    device: object
    stream: object      # torch.cuda.Stream every push of this stream runs on
    ring_len: int       # samples per channel: max(span of the first taps, history) + max_chunk
    n_chans: int | None = None
    on_device: bool | None = None
    ring: object = None
    d_in: object = None       # [header | block] as the kernel reads it
    stage_in: object = None   # pinned twin of d_in
    d_out: object = None
    stage_out: object = None
    graphs: dict = field(default_factory=dict)   # push shape -> captured CUDA graph
    seen: set = field(default_factory=set)       # push shapes run once eagerly
    lock: object = field(default_factory=threading.Lock)  # this stream's state, not the engine's


class DeviceEngine:
    """All GPU work of the PARRM hot path for one device."""

    def __init__(self, device: int | None = None):
        import torch

        if not torch.cuda.is_available() or _native.device_count() == 0:
            raise RuntimeError(
                "pyparrm_b200 needs an NVIDIA GPU (built for B200, sm_100a); no CUDA device is "
                "visible and there is no CPU fallback."
            )
        self.torch = torch
        index = torch.cuda.current_device() if device is None else int(device)
        self.device = torch.device("cuda", index)
        with torch.cuda.device(self.device):
            self.s_in = torch.cuda.Stream()
            self.s_run = torch.cuda.Stream()
            self.s_out = torch.cuda.Stream()
        self._lock = threading.RLock()
        self._count_lock = threading.Lock()  # the counters below; streams run outside _lock
        self._ring = None          # (key, slots)
        self._stage_in = None      # pinned staging for pageable inputs
        self._stage_out = None
        self._eval_ws = None
        self._plans: dict = {}
        self.launches = 0          # launches of ours enqueued: kernels + graph replays
        self.graph_kernels = 0     # kernels executed inside replayed CUDA graphs
        self.last_filter_kernel = ""

    # ------------------------------------------------------------------ helpers
    def _count(self, launches: int = 0, graph_kernels: int = 0) -> None:
        with self._count_lock:
            self.launches += launches
            self.graph_kernels += graph_kernels

    def _stream_ptr(self, stream) -> ctypes.c_void_p:
        return _vp(stream.cuda_stream)

    def _empty(self, n, dtype):
        return self.torch.empty(int(n), dtype=dtype, device=self.device)

    def _slots(self, in_bytes: int, out_bytes: int, x_bytes: int = 0, y_bytes: int = 0):
        """Device ring: per slot ``d_in`` (bytes as they arrive), ``d_out`` (bytes as they leave)
        and, when the storage type differs from the compute type, ``d_x`` / ``d_y``."""
        want = (in_bytes, out_bytes, x_bytes, y_bytes)
        if self._ring is None or any(h < w for h, w in zip(self._ring[0], want)):
            t = self.torch
            have = self._ring[0] if self._ring is not None else (0, 0, 0, 0)
            sizes = tuple(max(h, w) for h, w in zip(have, want))
            self._ring = None  # release the old ring before the new one is allocated
            slots = []
            for _ in range(_N_SLOTS):
                slots.append(
                    dict(
                        d_in=self._empty(max(sizes[0], 16), t.uint8),
                        d_out=self._empty(max(sizes[1], 16), t.uint8),
                        d_x=self._empty(max(sizes[2], 16), t.uint8),
                        d_y=self._empty(max(sizes[3], 16), t.uint8),
                        ev_in=t.cuda.Event(),
                        ev_run=t.cuda.Event(),
                        ev_out=t.cuda.Event(),
                        used=False,
                    )
                )
            self._ring = (sizes, slots)
        for slot in self._ring[1]:
            slot["used"] = False
        return self._ring[1]

    def _staging(self, which: str, nbytes: int):
        """Pinned host staging buffers (one per ring slot) for pageable arrays."""
        t = self.torch
        cur = getattr(self, which)
        if cur is None or cur[0].numel() < nbytes:
            cur = [t.empty(max(nbytes, 16), dtype=t.uint8, pin_memory=True) for _ in range(_N_SLOTS)]
            setattr(self, which, cur)
        return cur

    # ------------------------------------------------------------- period search
    def prepare_tiles(
        self, data: np.ndarray, index_sets: list[np.ndarray], outlier_boundary: float,
        precision: str = "fp64",
    ) -> list[SearchTile]:
        """Stream the recording through the device once: per-channel scale + gather.

        Restates ``_standardise_data`` (parrm.py:272-280) restricted to the columns the search
        reads (parrm.py:589-591), for every run's index set at once.
        """
        t = self.torch
        on_device = not isinstance(data, np.ndarray)
        if on_device:
            data, dtype_code = self._device_recording(data)
            elem = data.element_size()
        else:
            data, dtype_code = self._as_float_array(data, allow_f32=True)
            elem = data.dtype.itemsize
        n_chans, n_samples = data.shape
        with self._lock, t.cuda.device(self.device):
            tiles = []
            for idx in index_sets:
                idx = np.ascontiguousarray(idx, dtype=np.int64)
                if idx.size and (idx.min() < 0 or idx.max() > n_samples - 2):
                    raise IndexError("search indices outside the differenced recording")
                d_idx = t.from_numpy(idx).to(self.device)
                tiles.append(
                    SearchTile(
                        y=t.empty((idx.shape[0], n_chans), dtype=t.float64, device=self.device),
                        sumsq=t.empty(n_chans, dtype=t.float64, device=self.device),
                        indices=d_idx,
                        n_indices=int(idx.shape[0]),
                        n_chans=int(n_chans),
                    )
                )
            rows = max(1, _SEARCH_CHUNK_BYTES // max(1, n_samples * elem))
            rows = min(rows, n_chans, 65535)
            if on_device:
                self._device_tiles(data, rows, dtype_code, tiles, outlier_boundary)
                return self._fp32_tiles(tiles, precision)
            in_bytes = rows * n_samples * elem
            slots = self._slots(in_bytes, 16)
            ws_bytes = lib.parrm_channel_scales_workspace_bytes(rows, n_samples)
            scale = t.empty(n_chans, dtype=t.float64, device=self.device)
            ws = self._empty(max(ws_bytes, 16) * _N_SLOTS, t.uint8)
            pinned = is_pinned(data)
            stage = None if pinned else self._staging("_stage_in", in_bytes)
            run = self._stream_ptr(self.s_run)
            self.s_run.wait_stream(t.cuda.current_stream())
            for i, c0 in enumerate(range(0, n_chans, rows)):
                c1 = min(c0 + rows, n_chans)
                slot = slots[i % _N_SLOTS]
                nbytes = (c1 - c0) * n_samples * elem
                src = data.ctypes.data + c0 * n_samples * elem
                if slot["used"]:
                    slot["ev_run"].synchronize()  # kernels done with d_in (and staging reusable)
                if not pinned:
                    _threaded_memmove(stage[i % _N_SLOTS].data_ptr(), src, nbytes)
                    src = stage[i % _N_SLOTS].data_ptr()
                check(lib.parrm_copy_h2d_async(_vp(slot["d_in"].data_ptr()), _vp(src), nbytes,
                                               self._stream_ptr(self.s_in)), "H2D copy")
                slot["ev_in"].record(self.s_in)
                self.s_run.wait_event(slot["ev_in"])
                ws_ptr = ws.data_ptr() + (i % _N_SLOTS) * max(ws_bytes, 16)
                check(lib.parrm_channel_scales(
                    _vp(slot["d_in"].data_ptr()), c1 - c0, n_samples, n_samples,
                    _vp(scale.data_ptr() + 8 * c0), _vp(ws_ptr), ws_bytes, dtype_code, run),
                    "parrm_channel_scales")
                self._count(2)
                for tile in tiles:
                    check(lib.parrm_standardise_gather(
                        _vp(slot["d_in"].data_ptr()), c1 - c0, n_samples, n_samples,
                        _vp(tile.indices.data_ptr()), tile.n_indices,
                        _vp(scale.data_ptr() + 8 * c0), float(outlier_boundary),
                        _vp(tile.y.data_ptr() + 8 * c0), n_chans,
                        _vp(tile.sumsq.data_ptr() + 8 * c0), dtype_code, run),
                        "parrm_standardise_gather")
                    self._count(2)
                slot["ev_run"].record(self.s_run)
                slot["used"] = True
            self.s_run.synchronize()
            self._scale = scale
            return self._fp32_tiles(tiles, precision)

    def _fp32_tiles(self, tiles, precision):
        """float32 storage of the tiles in the fp32 mode; channel sums of the rounded values."""
        t = self.torch
        if precision == "fp32":
            with self._lock, t.cuda.device(self.device):
                sp = self._stream_ptr(t.cuda.current_stream())
                for tile in tiles:
                    tile.y = tile.y.to(t.float32)
                    check(lib.parrm_channel_sumsq(
                        _vp(tile.y.data_ptr()), _native.F32, tile.n_chans, tile.n_chans,
                        tile.n_indices, _vp(tile.sumsq.data_ptr()), sp), "parrm_channel_sumsq")
                    self._count(1)
                t.cuda.current_stream().synchronize()
        return tiles

    def _device_recording(self, data):
        """``(rows-contiguous [C, T] tensor, compute code)`` of a float64 / float32 CUDA recording
        on this engine's GPU (a row-strided view is copied to a dense tensor first)."""
        t = self.torch
        if data.device != self.device:
            raise ValueError(f"the recording is on {data.device}; this engine runs on {self.device}")
        code = {t.float64: _native.F64, t.float32: _native.F32}.get(data.dtype)
        if code is None:
            raise TypeError(f"unsupported data dtype {data.dtype}")
        if data.dim() != 2:
            raise ValueError("`data` must be a 2D array.")
        if not data.is_contiguous():
            data = data.contiguous()
        return data, code

    def _aligned_rows(self, data, c0: int, c1: int):
        """Channels ``[c0, c1)`` of a dense device recording, based at a 16-byte boundary as the
        host path's staging slots are (copied when the view's base is not): the scale kernel
        takes its vector loads, and with them its order of summation, only on aligned rows,
        so this is what keeps device and host results bit-equal."""
        block = data[c0:c1]
        return block if block.data_ptr() % 16 == 0 else block.clone()

    def _device_tiles(self, data, rows, dtype_code, tiles, outlier_boundary):
        """The device branch of :meth:`prepare_tiles`: the same channel blocks and row stride as
        the host path's staging slots, read where the recording lies (no H2D)."""
        t = self.torch
        n_chans, n_samples = data.shape
        sp = self._stream_ptr(t.cuda.current_stream())
        ws_bytes = lib.parrm_channel_scales_workspace_bytes(rows, n_samples)
        scale = t.empty(n_chans, dtype=t.float64, device=self.device)
        ws = self._empty(max(ws_bytes, 16), t.uint8)
        for c0 in range(0, n_chans, rows):
            c1 = min(c0 + rows, n_chans)
            block = self._aligned_rows(data, c0, c1)
            check(lib.parrm_channel_scales(
                _vp(block.data_ptr()), c1 - c0, n_samples, n_samples,
                _vp(scale.data_ptr() + 8 * c0), _vp(ws.data_ptr()), ws_bytes, dtype_code, sp),
                "parrm_channel_scales")
            self._count(2)
            for tile in tiles:
                check(lib.parrm_standardise_gather(
                    _vp(block.data_ptr()), c1 - c0, n_samples, n_samples,
                    _vp(tile.indices.data_ptr()), tile.n_indices,
                    _vp(scale.data_ptr() + 8 * c0), float(outlier_boundary),
                    _vp(tile.y.data_ptr() + 8 * c0), n_chans,
                    _vp(tile.sumsq.data_ptr() + 8 * c0), dtype_code, sp),
                    "parrm_standardise_gather")
                self._count(2)
        t.cuda.current_stream().synchronize()
        self._scale = scale

    def tile_from_standardised(self, z: np.ndarray, indices: np.ndarray) -> SearchTile:
        """Tile from an already standardised ``[channels, times]`` host array (the reference's
        ``_optimise_local(period, data, indices, ...)`` seam, parrm.py:552-559)."""
        t = self.torch
        indices = np.ascontiguousarray(indices, dtype=np.int64)
        y = np.ascontiguousarray(z[:, indices].T, dtype=np.float64)
        with self._lock, t.cuda.device(self.device):
            d_y = t.from_numpy(y).to(self.device)
            d_sumsq = t.empty(y.shape[1], dtype=t.float64, device=self.device)
            check(lib.parrm_channel_sumsq(_vp(d_y.data_ptr()), _native.F64, int(y.shape[1]),
                                          int(y.shape[1]), int(y.shape[0]), _vp(d_sumsq.data_ptr()),
                                          self._stream_ptr(t.cuda.current_stream())),
                  "parrm_channel_sumsq")
            self._count(1)
            return SearchTile(
                y=d_y, sumsq=d_sumsq, indices=t.from_numpy(indices).to(self.device),
                n_indices=int(y.shape[0]), n_chans=int(y.shape[1]),
            )

    def merge_channel_tiles(self, tile: SearchTile, all_gather, n_chans: int, per: int) -> SearchTile:
        """Tile of all ``n_chans`` channels from the per-rank tiles of channel blocks of ``per``
        channels (``_sharding.prepare_tiles_sharded``): the blocks are zero-padded to ``per``
        columns, exchanged with ``all_gather`` (-> ``[world, ...]``) and interleaved back into
        the sample-major ``[samples, channels]`` layout."""
        t = self.torch
        with self._lock, t.cuda.device(self.device):
            y = t.zeros((tile.n_indices, per), dtype=tile.y.dtype, device=self.device)
            y[:, : tile.n_chans] = tile.y
            sumsq = t.zeros(per, dtype=t.float64, device=self.device)
            sumsq[: tile.n_chans] = tile.sumsq
            ys = all_gather(y)              # [world, N, per]
            sums = all_gather(sumsq)        # [world, per]
            world = ys.shape[0]
            y_all = ys.permute(1, 0, 2).reshape(tile.n_indices, world * per)[:, :n_chans]
            return SearchTile(y=y_all.contiguous(), sumsq=sums.reshape(-1)[:n_chans].contiguous(),
                              indices=tile.indices, n_indices=tile.n_indices, n_chans=int(n_chans))

    def standardise_full(self, data: np.ndarray, outlier_boundary: float) -> np.ndarray:
        """The reference's ``_standard_data`` array [C, T-1] (parrm.py:272-280), on demand; a
        CUDA tensor for a CUDA recording."""
        t = self.torch
        on_device = not isinstance(data, np.ndarray)
        if on_device:  # a CUDA recording: read where it lies, a device tensor comes back
            data, dtype_code = self._device_recording(data)
            n_chans, n_samples = data.shape
            out = t.empty((n_chans, n_samples - 1), dtype=data.dtype, device=self.device)
            elem = data.element_size()
        else:
            data, dtype_code = self._as_float_array(data, allow_f32=True)
            n_chans, n_samples = data.shape
            out = np.empty((n_chans, n_samples - 1), dtype=data.dtype)
            elem = data.dtype.itemsize
        tdtype = t.float64 if dtype_code == _native.F64 else t.float32
        rows = max(1, min(n_chans, 65535, _CHUNK_BYTES // max(1, n_samples * elem)))
        with self._lock, t.cuda.device(self.device):
            stream = t.cuda.current_stream()
            sp = self._stream_ptr(stream)
            for c0 in range(0, n_chans, rows):
                c1 = min(c0 + rows, n_chans)
                if on_device:
                    d_x = self._aligned_rows(data, c0, c1)
                else:
                    d_x = t.from_numpy(np.ascontiguousarray(data[c0:c1])).to(self.device)
                scale = t.empty(c1 - c0, dtype=t.float64, device=self.device)
                ws_bytes = lib.parrm_channel_scales_workspace_bytes(c1 - c0, n_samples)
                ws = self._empty(max(ws_bytes, 16), t.uint8)
                check(lib.parrm_channel_scales(_vp(d_x.data_ptr()), c1 - c0, n_samples, n_samples,
                                               _vp(scale.data_ptr()), _vp(ws.data_ptr()), ws_bytes,
                                               dtype_code, sp), "parrm_channel_scales")
                d_z = t.empty((c1 - c0, n_samples - 1), dtype=tdtype, device=self.device)
                check(lib.parrm_standardise_full(_vp(d_x.data_ptr()), c1 - c0, n_samples,
                                                 n_samples, _vp(scale.data_ptr()),
                                                 float(outlier_boundary), _vp(d_z.data_ptr()),
                                                 n_samples - 1, dtype_code, sp),
                      "parrm_standardise_full")
                self._count(3)
                out[c0:c1] = d_z if on_device else d_z.cpu().numpy()
        return out

    def evaluate(
        self,
        tile: SearchTile,
        periods: np.ndarray,
        bandwidth: int,
        lambda_: float,
        n_chans_divisor: int,
    ) -> np.ndarray:
        """Objective of ``_optimise_local`` (parrm.py:552-597) for every candidate period."""
        periods = np.ascontiguousarray(periods, dtype=np.float64).ravel()
        n_periods = int(periods.shape[0])
        if n_periods == 0:
            return np.zeros(0, dtype=np.float64)
        d_err = self.evaluate_device(tile, periods, bandwidth, lambda_, n_chans_divisor)
        return d_err.cpu().numpy()

    def evaluate_device(self, tile, periods, bandwidth, lambda_, n_chans_divisor):
        """Like :meth:`evaluate`, but ``periods`` may be a device tensor and so is the result."""
        t = self.torch
        bandwidth = int(bandwidth)
        if bandwidth > _native.MAX_BANDWIDTH:
            raise ValueError(f"bandwidth {bandwidth} exceeds the device limit {_native.MAX_BANDWIDTH}")
        with self._lock, t.cuda.device(self.device):
            if isinstance(periods, np.ndarray):
                d_per = t.from_numpy(np.ascontiguousarray(periods, dtype=np.float64)).to(self.device)
            else:
                d_per = periods.to(device=self.device, dtype=t.float64).contiguous()
            n_periods = int(d_per.shape[0])
            d_err = t.empty(n_periods, dtype=t.float64, device=self.device)
            # One launch for the whole grid when its workspace fits (the sample splits, and with
            # them the workspace per candidate, shrink as the batch grows); otherwise halve.
            code = tile.y_code
            batch = n_periods
            while batch > 1 and lib.parrm_eval_workspace_bytes_typed(
                    tile.n_chans, tile.n_indices, batch, bandwidth, code) > _EVAL_WS_LIMIT:
                batch = -(-batch // 2)
            ws_bytes = max(
                lib.parrm_eval_workspace_bytes_typed(tile.n_chans, tile.n_indices, b, bandwidth, code)
                for b in {batch, n_periods % batch or batch}
            )
            if self._eval_ws is None or self._eval_ws.numel() < ws_bytes:
                self._eval_ws = self._empty(ws_bytes, t.uint8)
            sp = self._stream_ptr(t.cuda.current_stream())
            for p0 in range(0, n_periods, batch):
                p1 = min(p0 + batch, n_periods)
                need = lib.parrm_eval_workspace_bytes_typed(tile.n_chans, tile.n_indices, p1 - p0,
                                                            bandwidth, code)
                if self._eval_ws.numel() < need:
                    self._eval_ws = self._empty(need, t.uint8)
                self._count(self._eval_into(tile, d_per[p0:p1], d_err[p0:p1], bandwidth,
                                            lambda_, n_chans_divisor, sp))
            return d_err

    def _eval_into(self, tile, d_per, d_err, bandwidth, lambda_, n_chans_divisor, sp) -> int:
        """One parrm_eval_periods call on stream ``sp`` (no allocation: capturable); returns
        the number of kernels it enqueued."""
        n_periods = int(d_per.shape[0])
        code = tile.y_code
        check(lib.parrm_eval_periods_typed(
            _vp(tile.y.data_ptr()), code, tile.n_chans, _vp(tile.sumsq.data_ptr()),
            _vp(tile.indices.data_ptr()), tile.n_chans, tile.n_indices,
            _vp(d_per.data_ptr()), n_periods, int(bandwidth), float(lambda_),
            int(n_chans_divisor), _vp(d_err.data_ptr()),
            _vp(self._eval_ws.data_ptr()), self._eval_ws.numel(), sp), "parrm_eval_periods")
        if code == _native.F32:  # widened copy (dense float64 [N, C]) + the float64 kernels
            return 1 + lib.parrm_eval_launch_count(None, tile.n_chans, tile.n_chans,
                                                   tile.n_indices, n_periods, int(bandwidth))
        return lib.parrm_eval_launch_count(
            _vp(tile.y.data_ptr()), tile.n_chans, tile.n_chans, tile.n_indices, n_periods,
            int(bandwidth))

    ROUNDS_PER_GRAPH = 8

    def nm_minimise(self, tile, starts, bandwidth, lambda_, n_chans_divisor, xtol=1e-4,
                    ftol=1e-4, maxiter=200, maxfun=200):
        """``scipy.optimize.fmin`` (defaults) from every entry of ``starts`` on the objective of
        ``tile``, with the simplex state machines on the device (csrc/neldermead.cu): a round is
        one batched evaluation of 5 points per chain plus one state-machine step, and
        ``ROUNDS_PER_GRAPH`` rounds replay as one CUDA graph; the host reads one int32 per
        replay (chains still running) and the final states.  Returns ``[(x, fval, iterations,
        fcalls)]`` per chain, as ``fmin(..., full_output=True)[:4]``."""
        t = self.torch
        starts = np.ascontiguousarray(starts, dtype=np.float64).ravel()
        n = int(starts.shape[0])
        if n == 0:
            return []
        bandwidth = int(bandwidth)
        if bandwidth > _native.MAX_BANDWIDTH:
            raise ValueError(f"bandwidth {bandwidth} exceeds the device limit {_native.MAX_BANDWIDTH}")
        with self._lock, t.cuda.device(self.device):
            need = lib.parrm_eval_workspace_bytes_typed(tile.n_chans, tile.n_indices, 5 * n,
                                                        bandwidth, tile.y_code)
            if self._eval_ws is None or self._eval_ws.numel() < need:
                self._eval_ws = self._empty(need, t.uint8)
            d_starts = t.from_numpy(starts).to(self.device)
            d_state = t.zeros(n * _native.NM_STATE_BYTES, dtype=t.uint8, device=self.device)
            d_points = t.empty(5 * n, dtype=t.float64, device=self.device)
            d_values = t.empty(5 * n, dtype=t.float64, device=self.device)
            d_active = t.zeros(1, dtype=t.int32, device=self.device)
            kernels_per_round = [0]

            def one_round(sp):
                kernels_per_round[0] = 1 + self._eval_into(
                    tile, d_points, d_values, bandwidth, lambda_, n_chans_divisor, sp)
                check(lib.parrm_nm_step(
                    _vp(d_state.data_ptr()), n, _vp(d_values.data_ptr()), _vp(d_points.data_ptr()),
                    float(xtol), float(ftol), int(maxiter), int(maxfun),
                    _vp(d_active.data_ptr()), sp), "parrm_nm_step")

            stream = t.cuda.current_stream()
            sp = self._stream_ptr(stream)
            check(lib.parrm_nm_init(_vp(d_starts.data_ptr()), n, _vp(d_state.data_ptr()),
                                    _vp(d_points.data_ptr()), sp), "parrm_nm_init")
            one_round(sp)  # the initial simplex; also loads every kernel before the capture
            self._count(1 + kernels_per_round[0])
            active = int(d_active.item())
            if active:
                # capture_begin / capture_end directly: torch.cuda.graph() also runs
                # gc.collect() and empties the allocator cache, tens of ms per capture
                graph = t.cuda.CUDAGraph()
                self.s_run.wait_stream(stream)
                with t.cuda.stream(self.s_run):
                    graph.capture_begin(capture_error_mode="thread_local")
                    try:
                        for _ in range(self.ROUNDS_PER_GRAPH):
                            one_round(self._stream_ptr(self.s_run))
                    finally:
                        graph.capture_end()
                stream.wait_stream(self.s_run)
                replays = 0
                while active and replays * self.ROUNDS_PER_GRAPH < 2 * maxiter + 2:
                    graph.replay()
                    replays += 1
                    active = int(d_active.item())
                self._count(replays,            # one launch per replay ...
                            graph_kernels=replays * self.ROUNDS_PER_GRAPH * kernels_per_round[0])
            raw = d_state.cpu().numpy().view(np.dtype([
                ("sim", np.float64, 2), ("fsim", np.float64, 2), ("points", np.float64, 5),
                ("fcalls", np.int32), ("iterations", np.int32), ("done", np.int32),
                ("started", np.int32)]))
            return [(np.float64(r["sim"][0]), np.float64(np.min(r["fsim"])), int(r["iterations"]),
                     int(r["fcalls"])) for r in raw]

    def argmin(self, d_values):
        """(min value, first index) of a device vector, NaNs skipped (on device)."""
        t = self.torch
        with self._lock, t.cuda.device(self.device):
            d_val = t.empty(1, dtype=t.float64, device=self.device)
            d_idx = t.empty(1, dtype=t.int64, device=self.device)
            check(lib.parrm_argmin(_vp(d_values.data_ptr()), int(d_values.shape[0]),
                                   _vp(d_val.data_ptr()), _vp(d_idx.data_ptr()),
                                   self._stream_ptr(t.cuda.current_stream())), "parrm_argmin")
            self._count(1)
            return float(d_val.item()), int(d_idx.item())

    # --------------------------------------------------------------------- taps
    def build_taps(
        self, period: float, period_half_width: float, filter_half_width: int,
        omit_n_samples: int, direction: str,
    ) -> np.ndarray:
        """Tap offsets of ``_generate_filter`` (parrm.py:803-820), ascending int32."""
        t = self.torch
        with self._lock, t.cuda.device(self.device):
            d_taps = t.empty(2 * int(filter_half_width) + 1, dtype=t.int32, device=self.device)
            d_n = t.zeros(1, dtype=t.int32, device=self.device)
            check(lib.parrm_build_taps(
                float(period), float(period_half_width), int(filter_half_width),
                int(omit_n_samples), _native.DIRECTIONS[direction], _vp(d_taps.data_ptr()),
                _vp(d_n.data_ptr()), self._stream_ptr(t.cuda.current_stream())),
                "parrm_build_taps")
            self._count(1)
            n = int(d_n.item())
            return d_taps[:n].cpu().numpy()

    # ------------------------------------------------------------ parameter sweeps
    def default_half_widths(self, periods, period_half_widths, omits, limit: int) -> np.ndarray:
        """``_get_filter_half_width`` (parrm.py:788-801) for many parameter sets, one launch."""
        t = self.torch
        n = len(periods)
        with self._lock, t.cuda.device(self.device):
            d_per = t.tensor(np.asarray(periods, dtype=np.float64), device=self.device)
            d_phw = t.tensor(np.asarray(period_half_widths, dtype=np.float64), device=self.device)
            d_omit = t.tensor(np.asarray(omits, dtype=np.int64), device=self.device)
            d_lim = t.full((n,), int(limit), dtype=t.int64, device=self.device)
            d_out = t.empty(n, dtype=t.int64, device=self.device)
            check(lib.parrm_default_half_width(
                _vp(d_per.data_ptr()), _vp(d_phw.data_ptr()), _vp(d_omit.data_ptr()),
                _vp(d_lim.data_ptr()), n, _vp(d_out.data_ptr()),
                self._stream_ptr(t.cuda.current_stream())), "parrm_default_half_width")
            self._count(1)
            return d_out.cpu().numpy()

    def filter_sweep(self, data: np.ndarray, periods, period_half_widths, half_widths, omits,
                     directions):
        """Filter one recording with many tap sets: ONE tap-building launch and ONE filter
        launch for the whole sweep (``parrm_build_taps_batch`` -> ``parrm_filter_apply_batch``,
        the tap lists never leave the device in between).  Returns ``(out, taps)``: float64
        ``[n_sets, channels, times]`` and the per-set ascending tap offsets (an empty tap set
        -- the reference's RuntimeError, parrm.py:822-827 -- gives an empty array and zeros)."""
        t = self.torch
        data, code = self._as_float_array(data, allow_f32=False)
        n_sets = len(half_widths)
        n_chans, n_samples = data.shape
        max_hw = int(max(half_widths)) if n_sets else 1
        stride = 2 * max_hw + 1
        with self._lock, t.cuda.device(self.device):
            sp = self._stream_ptr(t.cuda.current_stream())
            dev = lambda a, dt: t.tensor(np.asarray(a, dtype=dt), device=self.device)  # noqa: E731
            d_per, d_phw = dev(periods, np.float64), dev(period_half_widths, np.float64)
            d_hw, d_omit = dev(half_widths, np.int64), dev(omits, np.int64)
            d_dir = dev([_native.DIRECTIONS[d] for d in directions], np.int32)
            d_taps = t.empty((n_sets, stride), dtype=t.int32, device=self.device)
            d_n = t.zeros(n_sets, dtype=t.int32, device=self.device)
            check(lib.parrm_build_taps_batch(
                _vp(d_per.data_ptr()), _vp(d_phw.data_ptr()), _vp(d_hw.data_ptr()),
                _vp(d_omit.data_ptr()), _vp(d_dir.data_ptr()), n_sets, _vp(d_taps.data_ptr()),
                stride, _vp(d_n.data_ptr()), sp), "parrm_build_taps_batch")
            d_x = t.from_numpy(data).to(self.device)
            d_out = t.empty((n_sets, n_chans, n_samples), dtype=t.float64, device=self.device)
            check(lib.parrm_filter_apply_batch(
                _vp(d_x.data_ptr()), n_samples, n_samples, n_chans, _vp(d_taps.data_ptr()), stride,
                _vp(d_n.data_ptr()), n_sets, max_hw, _vp(d_out.data_ptr()), n_samples,
                n_chans * n_samples, code, sp), "parrm_filter_apply_batch")
            self._count(2)
            self.last_filter_kernel = _native.filter_last_kernel()
            counts = d_n.cpu().numpy()
            taps_all = d_taps.cpu().numpy()
            return d_out.cpu().numpy(), [taps_all[i, : counts[i]].copy() for i in range(n_sets)]

    # -------------------------------------------------------------------- power
    def periodogram(self, data, n_points: int, sampling_freq: float) -> np.ndarray:
        """Base periodogram of ``compute_psd`` (``_utils/_power.py:63-66``) before its
        ``psd[:-1] *= 2``: float32 ``[channels, n_points // 2]`` (``[n_points // 2]`` for 1-D
        input).  ``data``: NumPy array (only the first ``n_points`` samples are uploaded) or a
        CUDA tensor (float64 / float32, rows contiguous)."""
        t = self.torch
        one_d = data.ndim == 1
        n_bins = int(n_points) // 2
        with self._lock, t.cuda.device(self.device):
            if isinstance(data, np.ndarray):
                head = np.atleast_2d(data)[:, : int(n_points)]
                head = np.ascontiguousarray(head, dtype=np.float32 if head.dtype != np.float64
                                            else np.float64)
                d_x = t.from_numpy(head).to(self.device)
            else:
                d_x = data if data.dim() == 2 else data.unsqueeze(0)
                if d_x.dtype not in (t.float64, t.float32) or d_x.stride(1) != 1:
                    d_x = d_x.to(t.float64).contiguous()
            code = _native.F64 if d_x.dtype == t.float64 else _native.F32
            n_chans, n_samples = d_x.shape
            d_psd = t.empty((n_chans, n_bins), dtype=t.float32, device=self.device)
            for c0 in range(0, n_chans, 65535):
                c1 = min(c0 + 65535, n_chans)
                check(lib.parrm_periodogram(
                    _vp(d_x[c0:c1].data_ptr()), c1 - c0, n_samples, d_x.stride(0), code,
                    int(n_points), float(sampling_freq), _vp(d_psd[c0:c1].data_ptr()), n_bins,
                    self._stream_ptr(t.cuda.current_stream())), "parrm_periodogram")
                self._count(1)
            psd = d_psd.cpu().numpy()
        return psd[0] if one_d else psd

    # ------------------------------------------------------------------- filter
    def _plan(self, taps: np.ndarray, dtype_code: int, strategy: int | None = None):
        """Host + device copies of the filter plan for a tap list (small LRU cache)."""
        t = self.torch
        taps = np.ascontiguousarray(taps, dtype=np.int32)
        if strategy is None:
            strategy = int(os.environ.get("PYPARRM_B200_PLAN", _native.PLAN_AUTO))
        key = (dtype_code, strategy, taps.tobytes())
        hit = self._plans.get(key)
        if hit is not None:
            return hit
        nbytes = lib.parrm_filter_plan_bytes(_vp(taps.ctypes.data), int(taps.shape[0]))
        h_plan = np.zeros(nbytes, dtype=np.uint8)
        check(lib.parrm_filter_plan(_vp(taps.ctypes.data), int(taps.shape[0]), dtype_code,
                                    int(strategy), _vp(h_plan.ctypes.data), nbytes),
              "parrm_filter_plan")
        d_plan = t.from_numpy(h_plan).to(self.device)
        if len(self._plans) >= 16:
            self._plans.pop(next(iter(self._plans)))
        span = (min(int(taps[0]), 0), max(int(taps[-1]), 0))
        self._plans[key] = (h_plan, d_plan, span)
        return self._plans[key]

    def _as_float_array(self, data: np.ndarray, allow_f32: bool):
        if data.dtype == np.float64:
            code = _native.F64
        elif data.dtype == np.float32 and allow_f32:
            code = _native.F32
        elif np.issubdtype(data.dtype, np.floating) or np.issubdtype(data.dtype, np.integer) \
                or data.dtype == np.bool_:
            data, code = data.astype(np.float64), _native.F64
        else:
            raise TypeError(f"unsupported data dtype {data.dtype}")
        if not data.flags.c_contiguous:
            data = np.ascontiguousarray(data)
        return data, code

    _STORAGE = {"float64": _native.F64, "float32": _native.F32, "int16": _native.I16,
                "int32": _native.I32}

    def _as_storage_array(self, data: np.ndarray):
        """``(C-contiguous array, storage code)``: float64 / float32 / int16 / int32 recordings
        are uploaded in their own width and widened on the device (the reference widens on the
        host, parrm.py:861-866); any other real dtype is first converted to float64 here."""
        code = self._STORAGE.get(data.dtype.name)
        if code is None:
            if not (np.issubdtype(data.dtype, np.floating) or np.issubdtype(data.dtype, np.integer)
                    or data.dtype == np.bool_):
                raise TypeError(f"unsupported data dtype {data.dtype}")
            data, code = data.astype(np.float64), _native.F64
        if not data.flags.c_contiguous:
            data = np.ascontiguousarray(data)
        return data, code

    # A job of at least this many channel-samples gets the kernel specialised for its plan
    # (built once per plan and device: ~0.5 s for the BASELINE tap sets); smaller one-off jobs
    # keep the pre-built kernels.  The build time grows faster than the unrolled step loop
    # (terms x box length loads per block: cfg2 200, 0.5 s; 860 taps in runs of 41: 1 764,
    # 22 s), so the job size that pays for it grows with the square of that.
    SPECIALISE_FROM = 1 << 24

    def _specialise_from(self, h_plan) -> int:
        info = np.zeros(16, dtype=np.int32)
        check(lib.parrm_filter_plan_info(_vp(h_plan.ctypes.data), _vp(info.ctypes.data), None, 0),
              "parrm_filter_plan_info")
        work = int(info[14]) * max(int(info[3]), int(info[4]), 1)  # terms x longest box
        return int(self.SPECIALISE_FROM * max(1.0, work / 400.0) ** 2)

    def _filter_options(self, job_samples: int, kernel=None, tuning=None, h_plan=None):
        opts = _native.FilterOptions()
        if kernel is None:
            kernel = int(os.environ.get("PYPARRM_B200_FILTER_KERNEL", _native.KERNEL_AUTO))
            threshold = self.SPECIALISE_FROM if h_plan is None else self._specialise_from(h_plan)
            if kernel == _native.KERNEL_AUTO and job_samples >= threshold:
                kernel = -1  # specialise when the plan allows, else whatever AUTO picks
        opts.kernel = _native.KERNEL_AUTO if kernel == -1 else int(kernel)
        opts.try_special = kernel == -1
        for name, value in (tuning or {}).items():
            setattr(opts, name, int(value))
        return opts

    def _apply(self, opts, *args):
        """parrm_filter_apply_ex; a job marked for specialisation tries that kernel first."""
        if opts.try_special:
            opts.kernel = _native.KERNEL_SPECIALISED
            status = lib.parrm_filter_apply_ex(*args[:-1], ctypes.byref(opts), args[-1])
            if status == 0:
                self.last_filter_kernel = _native.filter_last_kernel()
                return
            if status != 4:  # anything but "cannot specialise this plan / no NVRTC here"
                check(status, "parrm_filter_apply_ex")
            opts.kernel = _native.KERNEL_AUTO
            opts.try_special = False
        check(lib.parrm_filter_apply_ex(*args[:-1], ctypes.byref(opts), args[-1]),
              "parrm_filter_apply_ex")
        self.last_filter_kernel = _native.filter_last_kernel()

    def filter_device(self, d_x, taps: np.ndarray, d_out=None, stream=None, strategy=None,
                      kernel=None, tuning=None):
        """Filter a device-resident [C, T] tensor (float64 or float32); returns a device tensor."""
        t = self.torch
        code = {t.float64: _native.F64, t.float32: _native.F32}[d_x.dtype]
        if d_x.dim() != 2 or d_x.stride(1) != 1:
            raise ValueError("device input must be a 2-D row-major tensor")
        n_chans, n_samples = d_x.shape
        h_plan, d_plan, _ = self._plan(taps, code, strategy)
        if d_out is None:
            d_out = t.empty((n_chans, n_samples), dtype=d_x.dtype, device=d_x.device)
        stream = stream or t.cuda.current_stream()
        opts = self._filter_options(n_chans * n_samples, kernel, tuning, h_plan)
        for c0 in range(0, n_chans, 65535):
            c1 = min(c0 + 65535, n_chans)
            self._apply(
                opts, _vp(d_x[c0:c1].data_ptr()), d_x.stride(0), 0, n_samples,
                _vp(d_out[c0:c1].data_ptr()), d_out.stride(0), 0, n_samples, n_samples, c1 - c0,
                _vp(d_plan.data_ptr()), _vp(h_plan.ctypes.data), code, self._stream_ptr(stream))
            self._count(1)
        return d_out

    def filter_shard(self, chunk: np.ndarray, taps: np.ndarray, x0: int, t0: int, t1: int,
                     n_total: int, precision: str = "fp64"):
        """One shard of ``filter_data``, result left on the DEVICE (float64 ``[C, t1 - t0]``):
        ``chunk`` holds samples ``[x0, x0 + chunk.shape[1])`` of a recording of ``n_total``
        samples (the outputs' tap-window halo included); the outputs are those of global times
        ``[t0, t1)``.  Time shards (fewer channels than ranks) and the gather modes of
        ``enable_sharding`` use it: the shard goes on to a collective, not to the host."""
        t = self.torch
        chunk, _ = self._as_float_array(chunk, allow_f32=False)
        n_chans, n_x = chunk.shape
        f32 = precision == "fp32"
        code = _native.F32 if f32 else _native.F64
        with self._lock, t.cuda.device(self.device):
            h_plan, d_plan, _ = self._plan(taps, code)
            d_x = t.from_numpy(chunk).to(self.device)
            if f32:
                d_x = d_x.to(t.float32)
            d_out = t.empty((n_chans, t1 - t0), dtype=d_x.dtype, device=self.device)
            opts = self._filter_options(n_chans * (t1 - t0), h_plan=h_plan)
            for c0 in range(0, n_chans, 65535):
                c1 = min(c0 + 65535, n_chans)
                self._apply(
                    opts, _vp(d_x[c0:c1].data_ptr()), n_x, x0, n_x, _vp(d_out[c0:c1].data_ptr()),
                    t1 - t0, t0, t1 - t0, n_total, c1 - c0, _vp(d_plan.data_ptr()),
                    _vp(h_plan.ctypes.data), code, self._stream_ptr(t.cuda.current_stream()))
                self._count(1)
            return d_out.to(t.float64)

    def filter_host_window(self, chunk: np.ndarray, taps: np.ndarray, x0: int, t0: int, t1: int,
                           n_total: int) -> np.ndarray:
        """:meth:`filter_shard` with the result copied to the host."""
        return self.filter_shard(chunk, taps, x0, t0, t1, n_total).cpu().numpy()

    def filter_host(self, data: np.ndarray, taps: np.ndarray, precision: str = "fp64",
                    strategy: int | None = None, out_dtype=None) -> np.ndarray:
        """``filter_data`` body (parrm.py:861-869): NumPy [C, T] in, NumPy [C, T] out (float64
        as the reference returns it, or float32 on request).

        Bytes on PCIe: the recording goes up in the caller's dtype (float64, float32, int16 or
        int32) and is widened to the compute type on the device; the result comes back in
        ``out_dtype``.  ``precision="fp32"`` computes in float32."""
        t = self.torch
        data, in_code = self._as_storage_array(data)
        out_np = np.dtype(np.float64 if out_dtype is None else out_dtype)
        if out_np not in (np.dtype(np.float64), np.dtype(np.float32)):
            raise TypeError("`out_dtype` must be float64 or float32.")
        comp_code = _native.F32 if precision == "fp32" else _native.F64
        out_code = _native.F64 if out_np == np.float64 else _native.F32
        es_in, es_out = data.dtype.itemsize, out_np.itemsize
        es_c = 4 if comp_code == _native.F32 else 8
        n_chans, n_samples = data.shape
        out = self._output_array((n_chans, n_samples), out_np)
        if n_chans == 0 or n_samples == 0:
            return out
        with self._lock, t.cuda.device(self.device):
            h_plan, d_plan, (w_lo, w_hi) = self._plan(taps, comp_code, strategy)
            opts = self._filter_options(n_chans * n_samples, h_plan=h_plan)
            span = w_hi - w_lo
            row_bytes = n_samples * max(es_in, es_out)
            # chunk list: (c0, c1, t0, t1, x0, x1) -- channels [c0,c1), outputs [t0,t1), inputs [x0,x1)
            chunks = []
            if row_bytes <= 2 * _CHUNK_BYTES:
                rows = max(1, min(n_chans, 65535, _CHUNK_BYTES // row_bytes))
                for c0 in range(0, n_chans, rows):
                    chunks.append((c0, min(c0 + rows, n_chans), 0, n_samples, 0, n_samples))
            else:
                step = max(_CHUNK_BYTES // max(es_in, es_out), 4 * span)
                for c in range(n_chans):
                    for t0 in range(0, n_samples, step):
                        t1 = min(t0 + step, n_samples)
                        chunks.append((c, c + 1, t0, t1, max(0, t0 - w_hi), min(n_samples, t1 - w_lo)))
            in_elems = max((c1 - c0) * (x1 - x0) for c0, c1, _, _, x0, x1 in chunks)
            out_elems = max((c1 - c0) * (t1 - t0) for c0, c1, t0, t1, _, _ in chunks)
            widen_in, narrow_out = in_code != comp_code, comp_code != out_code
            slots = self._slots(in_elems * es_in, out_elems * es_out,
                                in_elems * es_c if widen_in else 0,
                                out_elems * es_c if narrow_out else 0)
            in_pinned, out_pinned = is_pinned(data), is_pinned(out)
            stage_in = None if in_pinned else self._staging("_stage_in", in_elems * es_in)
            stage_out = None if out_pinned else self._staging("_stage_out", out_elems * es_out)
            s_in, s_run, s_out = (self._stream_ptr(s) for s in (self.s_in, self.s_run, self.s_out))
            pending = [None] * _N_SLOTS  # (host dst ptr, nbytes) awaiting copy-out of staging

            def drain(k):
                if pending[k] is not None:
                    slots[k]["ev_out"].synchronize()
                    dst, nbytes = pending[k]
                    _threaded_memmove(dst, stage_out[k].data_ptr(), nbytes)
                    pending[k] = None

            for i, (c0, c1, t0, t1, x0, x1) in enumerate(chunks):
                k = i % _N_SLOTS
                slot = slots[k]
                n_c, n_x, n_o = c1 - c0, x1 - x0, t1 - t0
                src = data.ctypes.data + (c0 * n_samples + x0) * es_in
                dst = out.ctypes.data + (c0 * n_samples + t0) * es_out
                if slot["used"]:
                    if not in_pinned:
                        slot["ev_in"].synchronize()  # staging buffer free again
                    drain(k)
                n_in_bytes = n_c * n_x * es_in  # whole rows, or a time window of one row
                if not in_pinned:
                    _threaded_memmove(stage_in[k].data_ptr(), src, n_in_bytes)
                    src = stage_in[k].data_ptr()
                if slot["used"]:
                    self.s_in.wait_event(slot["ev_run"])   # kernel finished reading d_in
                check(lib.parrm_copy_h2d_async(_vp(slot["d_in"].data_ptr()), _vp(src),
                                               n_in_bytes, s_in), "H2D copy")
                slot["ev_in"].record(self.s_in)
                self.s_run.wait_event(slot["ev_in"])
                if slot["used"]:
                    self.s_run.wait_event(slot["ev_out"])  # previous result left d_out
                d_x = slot["d_in"].data_ptr()
                if widen_in:
                    check(lib.parrm_convert(_vp(d_x), in_code, _vp(slot["d_x"].data_ptr()),
                                            comp_code, n_c * n_x, s_run), "parrm_convert")
                    self._count(1)
                    d_x = slot["d_x"].data_ptr()
                d_y = slot["d_y"].data_ptr() if narrow_out else slot["d_out"].data_ptr()
                self._apply(
                    opts, _vp(d_x), n_x, x0, n_x, _vp(d_y), n_o, t0, n_o, n_samples,
                    n_c, _vp(d_plan.data_ptr()), _vp(h_plan.ctypes.data), comp_code, s_run)
                self._count(1)
                if narrow_out:
                    check(lib.parrm_convert(_vp(d_y), comp_code, _vp(slot["d_out"].data_ptr()),
                                            out_code, n_c * n_o, s_run), "parrm_convert")
                    self._count(1)
                slot["ev_run"].record(self.s_run)
                self.s_out.wait_event(slot["ev_run"])
                if out_pinned:
                    check(lib.parrm_copy_d2h_async(_vp(dst), _vp(slot["d_out"].data_ptr()),
                                                   n_c * n_o * es_out, s_out), "D2H copy")
                else:
                    check(lib.parrm_copy_d2h_async(_vp(stage_out[k].data_ptr()),
                                                   _vp(slot["d_out"].data_ptr()),
                                                   n_c * n_o * es_out, s_out), "D2H copy")
                    pending[k] = (dst, n_c * n_o * es_out)
                slot["ev_out"].record(self.s_out)
                slot["used"] = True
            for k in range(_N_SLOTS):
                drain(k)
            self.s_out.synchronize()
        return out

    # ------------------------------------------------------------- streaming
    # A stream's pushes take the stream's own lock, never the engine's ``_lock``: a period
    # search in another host thread (which holds ``_lock`` for each of its steps) must not
    # stall the acquisition loop.  They touch no shared engine state but the counters
    # (``_count``); ``parrm_host_copy`` serialises its callers itself.
    _STREAM_HEADER = 64      # bytes before the block in the staging buffers: {pos, out_lo}
    _STREAM_GRAPHS = 4       # captured push shapes kept per stream

    def stream_open(self, taps: np.ndarray, max_chunk: int, precision: str = "fp64",
                    history: int = 0):
        """State of one streaming filter (:mod:`pyparrm_b200._stream`): taps on the device, a
        CUDA stream of its own, and -- from the first push, which fixes the channel count -- the
        ring of the last ``max(span, history) + max_chunk`` samples per channel and pinned
        in/out staging.  Two streams never share any of it."""
        t = self.torch
        taps = np.ascontiguousarray(taps, dtype=np.int32)
        span = max(int(taps[-1]), 0) - min(int(taps[0]), 0)
        with t.cuda.device(self.device):
            return _StreamState(
                taps=taps, d_taps=t.from_numpy(taps).to(self.device), max_chunk=int(max_chunk),
                code=_native.F32 if precision == "fp32" else _native.F64,
                latency=max(0, -int(taps[0])), device=self.device,
                stream=t.cuda.Stream(device=self.device),
                ring_len=max(span, int(history)) + int(max_chunk))

    def stream_retune(self, st, taps: np.ndarray) -> None:
        """Switch an open stream to new taps (``FilterStream.set_filter``, which has checked
        that the ring holds what they read).  The upload runs on the stream's CUDA stream,
        after its pushes so far; the old tap tensor is kept until those have finished."""
        t = self.torch
        taps = np.ascontiguousarray(taps, dtype=np.int32)
        with st.lock, t.cuda.device(self.device):
            with t.cuda.stream(st.stream):
                d_taps = t.from_numpy(taps).to(self.device)
            st.d_taps.record_stream(st.stream)
            st.taps, st.d_taps, st.latency = taps, d_taps, max(0, -int(taps[0]))
            st.graphs.clear()
            st.seen.clear()

    def stream_recent(self, st, n: int, pos: int):
        """The last ``n`` of the ``pos`` samples pushed, ``[channels, n]`` in the compute type,
        copied out of the ring on the stream's CUDA stream (after its pushes); the caller's
        current stream waits for the copy."""
        t = self.torch
        with st.lock, t.cuda.device(self.device):
            comp = t.float32 if st.code == _native.F32 else t.float64
            out = t.empty((st.n_chans, int(n)), dtype=comp, device=self.device)
            current = t.cuda.current_stream()
            st.stream.wait_stream(current)
            check(lib.parrm_stream_window(
                _vp(st.ring.data_ptr()), st.ring_len, st.n_chans, int(pos), int(n),
                _vp(out.data_ptr()), int(n), st.code, self._stream_ptr(st.stream)),
                "parrm_stream_window")
            current.wait_stream(st.stream)
            return out

    def _stream_buffers(self, st, n_chans: int, in_bytes: int, out_bytes: int) -> None:
        """Ring at the first push; staging grown to the largest push (captured graphs hold the
        old pointers, so growing drops them)."""
        t = self.torch
        if st.ring is None:
            st.ring = self._empty(n_chans * st.ring_len * (4 if st.code == _native.F32 else 8),
                                  t.uint8)
            st.n_chans = n_chans
        in_bytes += self._STREAM_HEADER
        if st.d_in is None or st.d_in.numel() < in_bytes:
            st.d_in = self._empty(in_bytes, t.uint8)
            st.stage_in = t.empty(in_bytes, dtype=t.uint8, pin_memory=True)
            st.graphs.clear()
        if st.d_out is None or st.d_out.numel() < max(out_bytes, 16):
            st.d_out = self._empty(max(out_bytes, 16), t.uint8)
            st.stage_out = t.empty(max(out_bytes, 16), dtype=t.uint8, pin_memory=True)
            st.graphs.clear()

    def _stream_launch(self, st, d_block, block_code, ld_block, n, d_out, out_code, k, pos,
                       out_lo, d_hdr, close, sp) -> None:
        w_min, w_max = int(st.taps[0]), int(st.taps[-1])
        check(lib.parrm_stream_push_at(
            _vp(st.ring.data_ptr()), st.ring_len, st.n_chans, _vp(st.d_taps.data_ptr()),
            int(st.taps.shape[0]), w_min, w_max, _vp(d_block), block_code, ld_block, n,
            _vp(d_out), out_code, max(k, 1), pos, out_lo, d_hdr, int(close), st.code, sp),
            "parrm_stream_push_at")

    def stream_push(self, st, block, pos: int, close: bool, out_dtype=None, graphs: bool = False,
                    emitted: int | None = None):
        """One push (``block`` None: nothing new, the closing push): returns the outputs it makes
        final, ``_stream.output_range`` (from ``emitted``, the outputs returned so far, once the
        stream's taps have been switched).  NumPy blocks go through the stream's pinned staging
        (H2D, one kernel, D2H, on the stream's own CUDA stream); with ``graphs``, a push of the
        same shape as an earlier one that returns exactly one output per sample is captured
        once and then replayed as one CUDA graph that reads the positions from a header copied
        up with the block.  CUDA blocks are read where they lie and a CUDA tensor comes back."""
        from ._stream import output_range

        t = self.torch
        with st.lock, t.cuda.device(self.device):
            if st.on_device is None:
                st.on_device = block is not None and not isinstance(block, np.ndarray)
            if st.on_device:
                return self._stream_push_device(st, block, pos, close, emitted, output_range)
            if block is None:
                block = np.zeros((st.n_chans, 0), dtype=np.float64)
            data, in_code = self._as_storage_array(block)
            n_chans, n = data.shape
            out_np = np.dtype(np.float64 if out_dtype is None else out_dtype)
            out_code = _native.F64 if out_np == np.float64 else _native.F32
            lo, hi = output_range(pos, n, st.latency, close, emitted)
            k = hi - lo
            in_bytes, out_bytes = data.nbytes, n_chans * k * out_np.itemsize
            self._stream_buffers(st, n_chans, in_bytes, out_bytes)
            hdr = self._STREAM_HEADER
            d_in, h_in = st.d_in.data_ptr(), st.stage_in.data_ptr()
            d_out, h_out = st.d_out.data_ptr(), st.stage_out.data_ptr()
            if in_bytes:
                _threaded_memmove(h_in + hdr, data.ctypes.data, in_bytes)
            sp = self._stream_ptr(st.stream)
            key = (n_chans, n, in_code, out_code)
            replayable = graphs and not close and k == n and n > 0
            if replayable and (key in st.graphs or key in st.seen):
                st.stage_in[:16].numpy().view(np.int64)[:] = (pos, lo)
                graph = st.graphs.get(key)
                if graph is None:
                    graph = self._stream_capture(st, key, data.shape, in_code, out_code, k, pos,
                                                 lo)
                with t.cuda.stream(st.stream):
                    graph.replay()
                self._count(1, graph_kernels=1)
            else:
                check(lib.parrm_copy_h2d_async(_vp(d_in + hdr), _vp(h_in + hdr), in_bytes, sp),
                      "H2D copy")
                self._stream_launch(st, d_in + hdr, in_code, n, n, d_out, out_code, k, pos, lo,
                                    None, close, sp)
                self._count(1)
                check(lib.parrm_copy_d2h_async(_vp(h_out), _vp(d_out), out_bytes, sp), "D2H copy")
                if replayable:
                    st.seen.add(key)
            st.stream.synchronize()
            view = st.stage_out[:out_bytes].numpy().view(out_np).reshape(n_chans, k)
            return view.copy()

    def _stream_capture(self, st, key, shape, in_code, out_code, k, pos, lo):
        """Capture H2D (header + block) -> kernel -> D2H of a push shape as one CUDA graph."""
        t = self.torch
        n_chans, n = shape
        es_in = {_native.F64: 8, _native.F32: 4, _native.I16: 2, _native.I32: 4}[in_code]
        es_out = 8 if out_code == _native.F64 else 4
        hdr = self._STREAM_HEADER
        d_in, h_in = st.d_in.data_ptr(), st.stage_in.data_ptr()
        d_out, h_out = st.d_out.data_ptr(), st.stage_out.data_ptr()
        graph = t.cuda.CUDAGraph()
        with t.cuda.stream(st.stream):
            sp = self._stream_ptr(st.stream)
            graph.capture_begin(capture_error_mode="thread_local")
            try:
                check(lib.parrm_copy_h2d_async(_vp(d_in), _vp(h_in), hdr + n_chans * n * es_in, sp),
                      "H2D copy")
                self._stream_launch(st, d_in + hdr, in_code, n, n, d_out, out_code, k, pos, lo,
                                    _vp(d_in), False, sp)
                check(lib.parrm_copy_d2h_async(_vp(h_out), _vp(d_out), n_chans * k * es_out, sp),
                      "D2H copy")
            finally:
                graph.capture_end()
        if len(st.graphs) >= self._STREAM_GRAPHS:
            st.graphs.pop(next(iter(st.graphs)))
        st.graphs[key] = graph
        return graph

    _TORCH_STORAGE = {"torch.float64": _native.F64, "torch.float32": _native.F32,
                      "torch.int16": _native.I16, "torch.int32": _native.I32}

    def _stream_push_device(self, st, block, pos, close, emitted, output_range):
        t = self.torch
        comp = t.float32 if st.code == _native.F32 else t.float64
        if block is None:
            block = t.empty((st.n_chans, 0), dtype=comp, device=self.device)
        code = self._TORCH_STORAGE.get(str(block.dtype))
        if code is None:
            block, code = block.to(t.float64), _native.F64
        if block.stride(1) != 1 and block.shape[1] > 1:
            block = block.contiguous()
        n_chans, n = block.shape
        lo, hi = output_range(pos, n, st.latency, close, emitted)
        self._stream_buffers(st, n_chans, 0, 0)
        out = t.empty((n_chans, hi - lo), dtype=comp, device=self.device)
        current = t.cuda.current_stream()
        st.stream.wait_stream(current)
        self._stream_launch(st, block.data_ptr(), code, max(block.stride(0), n), n, out.data_ptr(),
                            st.code, hi - lo, pos, lo, None, close, self._stream_ptr(st.stream))
        self._count(1)
        current.wait_stream(st.stream)
        return out

    # Results are handed to the caller in page-locked memory (direct D2H, no staging copy) up
    # to this many live bytes; beyond that -- many results kept alive, or huge ones -- they are
    # ordinary pageable arrays filled through the pinned staging ring, so a caller can never
    # page-lock more than the limit through this path.  torch's host allocator caches freed
    # pinned blocks; when a result of a new size would push the cache past the limit the
    # cache is emptied first.
    def _output_array(self, shape, dtype) -> np.ndarray:
        import weakref

        nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        live = getattr(self, "_pinned_live", 0)
        if nbytes == 0 or live + nbytes > _PINNED_OUT_LIMIT:
            return np.empty(shape, dtype=dtype)
        if nbytes not in getattr(self, "_pinned_sizes", set()):
            sizes = getattr(self, "_pinned_sizes", set())
            if sum(sizes) + nbytes > _PINNED_OUT_LIMIT:
                empty_cache = getattr(self.torch._C, "_host_emptyCache", None)
                if empty_cache is not None:
                    empty_cache()
                sizes.clear()
            sizes.add(nbytes)
            self._pinned_sizes = sizes
        out = pinned_empty(shape, dtype)
        self._pinned_live = live + nbytes
        weakref.finalize(out.base if out.base is not None else out, self._release_pinned, nbytes)
        return out

    def _release_pinned(self, nbytes: int) -> None:
        self._pinned_live = max(0, getattr(self, "_pinned_live", 0) - nbytes)


_engine: DeviceEngine | None = None
_engine_lock = threading.Lock()


def get_engine() -> DeviceEngine:
    """Process-wide engine for the current CUDA device (created on first use)."""
    global _engine
    with _engine_lock:
        if _engine is None:
            _engine = DeviceEngine()
        return _engine


def current_engine():
    """The process-wide engine if one exists already (never creates it)."""
    return _engine


def set_engine(engine) -> None:
    """Install an engine object (tests inject a stand-in; ``None`` resets)."""
    global _engine
    with _engine_lock:
        _engine = engine

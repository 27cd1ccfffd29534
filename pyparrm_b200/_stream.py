"""Streaming filter: ``PARRM.filter_stream()``, the filter applied block by block as a recording
is acquired.

An online caller runs ``find_period()`` and ``create_filter()`` on a calibration segment, then
pushes every block the acquisition system delivers::

    stream = parrm.filter_stream()
    for block in acquisition:          # [channels, n]: NumPy array or CUDA tensor
        y = stream.push(block)         # [channels, k]: every output that is now final
    tail = stream.close()              # the last `stream.latency` outputs

Concatenating every ``push()`` result and ``close()`` gives exactly ``filter_data()`` on the
concatenated recording, start and end edges and the non-finite rule included.  Output ``t`` is
final once sample ``t + latency`` has arrived.  Under the reference's convolution ``y[t]``
reads ``x[t - w]`` for the taps ``w``, so a ``"future"`` filter (``w > 0``) reads only earlier
samples and has latency 0: it is the causal direction.  ``"past"`` and ``"both"`` need up to
``filter_half_width`` samples of look-ahead.

The artefact period can change during an online session (the stimulation is reprogrammed, the
stimulator and amplifier clocks drift apart).  A stream opened with ``history`` keeps that many
recent samples on the device; ``recent(n)`` hands them out as a CUDA tensor to re-run
``find_period()`` on, and ``set_filter(parrm)`` switches the stream to the new taps without a
gap or a repeated output::

    stream = parrm.filter_stream(history=10 * fs)
    for block in acquisition:
        y = stream.push(block)
        if settings_changed:
            cal = PARRM(stream.recent(10 * fs), fs, new_fa, verbose=False)
            cal.find_period(); cal.create_filter(filter_direction="future")
            stream.set_filter(cal)     # every output not yet returned uses the new taps

This module holds the bookkeeping (positions, output ranges, validation, splitting of long
blocks, the switch point); the engine owns the per-stream device state and runs the kernel
(``DeviceEngine.stream_open`` / ``stream_push`` / ``stream_retune`` / ``stream_recent``, one
launch per push).
"""

from __future__ import annotations

import threading

import numpy as np

_CLOSED_MSG = "This stream has been closed."


def output_range(pos: int, n: int, latency: int, close: bool,
                 emitted: int | None = None) -> tuple[int, int]:
    """Outputs ``[lo, hi)`` a push of ``n`` samples at position ``pos`` makes final: those whose
    taps have all arrived, or, on the closing push, all that are left.  ``lo`` is ``emitted``,
    the outputs returned so far, when given; without it, ``max(0, pos - latency)``, which is
    the same number as long as the stream has had one tap set."""
    lo = max(0, pos - latency) if emitted is None else int(emitted)
    hi = pos + n if close else max(lo, pos + n - latency)
    return lo, hi


def _span(taps) -> int:
    return max(int(taps[-1]), 0) - min(int(taps[0]), 0)


def _is_device_tensor(obj) -> bool:
    return (type(obj).__module__.split(".")[0] == "torch" and hasattr(obj, "is_cuda")
            and bool(obj.is_cuda))


class FilterStream:
    """A filter applied to a recording that arrives in consecutive blocks.

    Made by :meth:`pyparrm_b200.PARRM.filter_stream`, which snapshots the filter's taps and
    the object's precision: a later ``create_filter()`` does not change an open stream; only
    :meth:`set_filter` switches its taps.

    Attributes
    ----------
    latency : int
        ``max(0, -min(taps))`` of the current taps: output ``t`` comes out of the push that
        delivers sample ``t + latency`` (0 for ``filter_direction="future"``).
    n_pushed : int
        Samples pushed so far.
    n_emitted : int
        Outputs returned so far.
    history : int
        Samples per channel the device ring keeps beyond what filtering needs, for
        :meth:`recent` (0: none).
    """

    def __init__(self, engine, taps, precision: str = "fp64", max_chunk: int = 1 << 16,
                 out_dtype=None, graphs: bool = False, history: int = 0):
        if not isinstance(max_chunk, (int, np.integer)) or isinstance(max_chunk, bool):
            raise TypeError("`max_chunk` must be an int.")
        if max_chunk < 1:
            raise ValueError("`max_chunk` must be >= 1.")
        if not isinstance(history, (int, np.integer)) or isinstance(history, bool):
            raise TypeError("`history` must be an int.")
        if history < 0:
            raise ValueError("`history` must be >= 0.")
        out_np = np.dtype(np.float64 if out_dtype is None else out_dtype)
        if out_np not in (np.dtype(np.float64), np.dtype(np.float32)):
            raise TypeError("`out_dtype` must be float64 or float32.")
        taps = np.array(taps, dtype=np.int32, copy=True)
        if taps.ndim != 1 or taps.shape[0] == 0 or np.any(np.diff(taps) <= 0):
            raise ValueError("the taps must be a non-empty ascending list of offsets")
        self._engine = engine
        self._taps = taps
        self._precision = precision
        self._out_dtype = out_np
        self.max_chunk = int(max_chunk)
        self.graphs = bool(graphs)
        self.latency = max(0, -int(taps[0]))
        self.history = int(history)
        # samples per channel of the device ring: what the pushes read, and the history
        self.ring_len = max(_span(taps), self.history) + self.max_chunk
        if self.history:
            self._state = engine.stream_open(taps, self.max_chunk, precision,
                                             history=self.history)
        else:
            self._state = engine.stream_open(taps, self.max_chunk, precision)
        self._n_chans = None
        self._on_device = None
        self._closed = False
        self._switched = False  # the taps changed: the first output comes from n_emitted
        self._lock = threading.RLock()
        self.n_pushed = 0
        self.n_emitted = 0

    @property
    def taps(self) -> np.ndarray:
        """The tap offsets this stream filters with (a copy)."""
        return self._taps.copy()

    def _check_block(self, block):
        on_device = _is_device_tensor(block)
        if not on_device and not isinstance(block, np.ndarray):
            raise TypeError("`block` must be a NumPy array or a CUDA tensor.")
        if block.ndim != 2:
            raise ValueError("`block` must be a 2D array.")
        n_chans = int(block.shape[0])
        if self._n_chans is None:
            self._n_chans, self._on_device = n_chans, on_device
        elif n_chans != self._n_chans:
            raise ValueError(
                f"`block` has {n_chans} channels; this stream was started with {self._n_chans}.")
        elif on_device != self._on_device:
            raise TypeError("A stream is fed either NumPy arrays or CUDA tensors, not both.")
        return on_device

    def _empty(self, n_chans: int, block=None):
        if self._on_device:
            import torch

            dtype = torch.float32 if self._precision == "fp32" else torch.float64
            return torch.empty((n_chans, 0), dtype=dtype, device=block.device if block is not None
                               else self._state.device)
        return np.zeros((n_chans, 0), dtype=self._out_dtype)

    def _run(self, block, close: bool):
        n = 0 if block is None else int(block.shape[1])
        emitted = {"emitted": self.n_emitted} if self._switched else {}
        lo, hi = output_range(self.n_pushed, n, self.latency, close, **emitted)
        out = self._engine.stream_push(self._state, block, self.n_pushed, close,
                                       out_dtype=self._out_dtype, graphs=self.graphs, **emitted)
        if out.shape[1] != hi - lo:
            raise RuntimeError(f"stream kernel returned {out.shape[1]} outputs, expected {hi - lo}")
        self.n_pushed += n
        self.n_emitted = hi
        return out

    def push(self, block):
        """Filter the next ``[channels, n]`` block (NumPy float64 / float32 / int16 / int32 --
        other real dtypes are converted to float64 -- or a CUDA tensor) and return every output
        that is now final: ``[channels, k]``, NumPy in ``out_dtype`` for NumPy blocks, a CUDA
        tensor in the compute type for CUDA blocks.  Blocks longer than ``max_chunk`` are split
        here; the channel count is fixed by the first push."""
        with self._lock:
            return self._push(block)

    def _push(self, block):
        if self._closed:
            raise RuntimeError(_CLOSED_MSG)
        on_device = self._check_block(block)
        n = int(block.shape[1])
        if n == 0:
            return self._empty(self._n_chans, block)
        if n <= self.max_chunk:
            return self._run(block, close=False)
        parts = [self._run(block[:, s:s + self.max_chunk], close=False)
                 for s in range(0, n, self.max_chunk)]
        if on_device:
            import torch

            return torch.cat(parts, dim=1)
        return np.concatenate(parts, axis=1)

    def close(self):
        """End the recording: return the outputs still held back (the last ``latency``, or
        fewer when less was pushed), computed with the recording-end edge."""
        with self._lock:
            return self._close()

    def _close(self):
        if self._closed:
            raise RuntimeError(_CLOSED_MSG)
        self._closed = True
        if self._n_chans is None:  # nothing was pushed
            return np.zeros((0, 0), dtype=self._out_dtype)
        if self.n_emitted == self.n_pushed:
            return self._empty(self._n_chans)
        return self._run(None, close=True)

    def recent(self, n: int):
        """The last ``n`` samples pushed, ``[channels, n]``, as a CUDA tensor in the compute type
        (float64, or float32 for an fp32 stream): the values the device ring holds, widened from
        the blocks' storage type exactly as the filter reads them -- for NumPy-fed streams too.
        Needs ``1 <= n <= min(n_pushed, history)``.  The copy is ordered after the last push and
        the caller's current CUDA stream waits for it; nothing crosses PCIe.

        Hand the window to ``PARRM(stream.recent(n), fs, fa)`` to re-estimate the period on the
        GPU, then :meth:`set_filter` the result."""
        with self._lock:
            if self._closed:
                raise RuntimeError(_CLOSED_MSG)
            if not isinstance(n, (int, np.integer)) or isinstance(n, bool):
                raise TypeError("`n` must be an int.")
            if not 1 <= n <= min(self.n_pushed, self.history):
                raise ValueError(
                    f"recent({n}): `n` must lie in [1, min(samples pushed = {self.n_pushed}, "
                    f"history = {self.history})]; open the stream with "
                    f"filter_stream(history=...) of at least the window you need.")
            return self._engine.stream_recent(self._state, int(n), self.n_pushed)

    def set_filter(self, parrm) -> None:
        """Switch to the current filter of ``parrm`` (a :class:`pyparrm_b200.PARRM` after
        ``create_filter()``; only its taps are taken -- the stream keeps its precision).

        The switch point is ``s = n_emitted``: every output already returned was computed with
        the old taps, every later one with the new, so all pushes plus ``close()`` concatenate
        to ``filter_data()`` of the whole recording with each tap set over its own range of
        outputs (start and end edges those of the whole recording).  ``latency`` becomes that of
        the new taps; captured CUDA graphs are dropped.  The ring must hold both the new taps'
        span and what the outputs still pending reach back to,
        ``(n_pushed - n_emitted) + max(0, max(taps))``; otherwise ``ValueError``, naming the
        ``history`` that would make it fit."""
        if getattr(parrm, "_filter", None) is None:
            raise ValueError(
                "The filter has not yet been created. The `create_filter` method must "
                "be called first."
            )
        taps = np.ascontiguousarray(parrm._tap_offsets(), dtype=np.int32)
        with self._lock:
            if self._closed:
                raise RuntimeError(_CLOSED_MSG)
            reach = (self.n_pushed - self.n_emitted) + max(int(taps[-1]), 0)
            need = max(_span(taps), reach)
            if need > self.ring_len - self.max_chunk:
                raise ValueError(
                    f"The new filter needs {need} samples per channel in the stream's ring (tap "
                    f"span {_span(taps)}, pending outputs reach back {reach}); it holds "
                    f"{self.ring_len - self.max_chunk}.  Open the stream with "
                    f"filter_stream(history={need}) or more.")
            self._engine.stream_retune(self._state, taps)
            self._taps = taps
            self.latency = max(0, -int(taps[0]))
            self._switched = True

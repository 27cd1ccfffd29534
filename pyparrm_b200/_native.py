"""ctypes binding of ``libparrm_b200.so`` (C ABI declared in ``include/parrm_b200.h``).

The library is built in-tree by ``pyparrm_b200/csrc/build.sh`` (``__graft_entry__.build``).
There is no fallback: if the shared object is missing, importing this module raises, and
every compute entry point raises ``RuntimeError`` with the library's own message when the
CUDA call behind it fails (e.g. on a host without a GPU).
"""

from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_int, c_int32, c_int64, c_size_t, c_void_p

LIB_NAME = "libparrm_b200.so"
LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), LIB_NAME)

F64, F32, I16, I32 = 0, 1, 2, 3
DIR_BOTH, DIR_PAST, DIR_FUTURE = 0, 1, 2
DIRECTIONS = {"both": DIR_BOTH, "past": DIR_PAST, "future": DIR_FUTURE}
MAX_BANDWIDTH = 23
NM_STATE_BYTES = 88
ABI_VERSION = 8
PLAN_AUTO, PLAN_GATHER, PLAN_COMB = 0, 1, 2
KERNEL_AUTO, KERNEL_GATHER, KERNEL_SPECIALISED = 0, 1, 3


class FilterOptions(ctypes.Structure):
    """``parrm_filter_options_t`` (include/parrm_b200.h); all zero = library defaults."""

    _fields_ = [
        ("kernel", c_int32),
        ("steps_per_chunk", c_int32),
        ("prefetch_chunks", c_int32),
        ("ctas_per_sm", c_int32),
        ("variant", c_int32),
        ("reserved", c_int32),
        ("timeline", ctypes.c_uint64),
    ]


# name -> (restype, argtypes); mirrors include/parrm_b200.h one to one
SIGNATURES = {
    "parrm_abi_version": (c_int, []),
    "parrm_last_error": (c_char_p, []),
    "parrm_device_count": (c_int, []),
    "parrm_host_is_pinned": (c_int, [c_void_p]),
    "parrm_copy_h2d_async": (c_int, [c_void_p, c_void_p, c_size_t, c_void_p]),
    "parrm_copy_d2h_async": (c_int, [c_void_p, c_void_p, c_size_t, c_void_p]),
    "parrm_channel_scales_workspace_bytes": (c_size_t, [c_int64, c_int64]),
    "parrm_channel_scales": (
        c_int,
        [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_void_p, c_size_t, c_int, c_void_p],
    ),
    "parrm_standardise_gather": (
        c_int,
        [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_double,
         c_void_p, c_int64, c_void_p, c_int, c_void_p],
    ),
    "parrm_channel_sumsq": (
        c_int, [c_void_p, c_int, c_int64, c_int64, c_int64, c_void_p, c_void_p]),
    "parrm_eval_workspace_bytes_typed": (c_size_t, [c_int64, c_int64, c_int64, c_int, c_int]),
    "parrm_eval_periods_typed": (
        c_int,
        [c_void_p, c_int, c_int64, c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_int64, c_int,
         c_double, c_int64, c_void_p, c_void_p, c_size_t, c_void_p],
    ),
    "parrm_standardise_full": (
        c_int,
        [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_double, c_void_p, c_int64, c_int,
         c_void_p],
    ),
    "parrm_eval_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64, c_int]),
    "parrm_eval_launch_count": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_int64, c_int]),
    "parrm_eval_periods": (
        c_int,
        [c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_int64, c_int,
         c_double, c_int64, c_void_p, c_void_p, c_size_t, c_void_p],
    ),
    "parrm_argmin": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "parrm_build_taps": (
        c_int, [c_double, c_double, c_int64, c_int64, c_int, c_void_p, c_void_p, c_void_p]
    ),
    "parrm_filter_plan_bytes": (c_size_t, [c_void_p, c_int32]),
    "parrm_filter_plan": (c_int, [c_void_p, c_int32, c_int, c_int, c_void_p, c_size_t]),
    "parrm_filter_plan_info": (c_int, [c_void_p, c_void_p, c_void_p, c_int32]),
    "parrm_filter_apply": (
        c_int,
        [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int64, c_int64, c_int64, c_int64,
         c_int64, c_void_p, c_void_p, c_int, c_void_p],
    ),
    "parrm_filter_apply_ex": (
        c_int,
        [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int64, c_int64, c_int64, c_int64,
         c_int64, c_void_p, c_void_p, c_int, POINTER(FilterOptions), c_void_p],
    ),
    "parrm_filter_last_kernel": (c_char_p, []),
    "parrm_filter_specialise_check": (
        c_int, [c_void_p, c_int, POINTER(FilterOptions), c_void_p, POINTER(c_size_t)]
    ),
    "parrm_host_register": (c_int, [c_void_p, c_size_t]),
    "parrm_host_unregister": (c_int, [c_void_p]),
    "parrm_host_copy": (c_int, [c_void_p, c_void_p, c_size_t, c_int]),
    "parrm_convert": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int64, c_void_p]),
    "parrm_convert_f64_to_f32": (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    "parrm_convert_f32_to_f64": (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    "parrm_nm_init": (c_int, [c_void_p, c_int32, c_void_p, c_void_p, c_void_p]),
    "parrm_nm_step": (
        c_int,
        [c_void_p, c_int32, c_void_p, c_void_p, c_double, c_double, c_int32, c_int32, c_void_p,
         c_void_p]),
    "parrm_default_half_width": (
        c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "parrm_build_taps_batch": (
        c_int,
        [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_void_p,
         c_void_p]),
    "parrm_filter_apply_batch": (
        c_int,
        [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_int64, c_int64,
         c_void_p, c_int64, c_int64, c_int, c_void_p]),
    "parrm_periodogram": (
        c_int,
        [c_void_p, c_int64, c_int64, c_int64, c_int, c_int64, c_double, c_void_p, c_int64, c_void_p],
    ),
    "parrm_stream_ring_bytes": (c_size_t, [c_int64, c_void_p, c_int32, c_int64, c_int]),
    "parrm_stream_push": (
        c_int,
        [c_void_p, c_int64, c_int64, c_void_p, c_int32, c_int32, c_int32, c_void_p, c_int,
         c_int64, c_int64, c_void_p, c_int, c_int64, c_int64, c_void_p, c_int, c_int, c_void_p],
    ),
    "parrm_stream_push_at": (
        c_int,
        [c_void_p, c_int64, c_int64, c_void_p, c_int32, c_int32, c_int32, c_void_p, c_int,
         c_int64, c_int64, c_void_p, c_int, c_int64, c_int64, c_int64, c_void_p, c_int, c_int,
         c_void_p],
    ),
    "parrm_stream_window": (
        c_int, [c_void_p, c_int64, c_int64, c_int64, c_int64, c_void_p, c_int64, c_int, c_void_p]),
    "parrm_fp64_fma_burn": (c_int, [c_int64, c_void_p, POINTER(c_double), c_void_p]),
}


def _load() -> ctypes.CDLL:
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_NAME} is not built (expected {LIB_PATH}). Build it with "
            "`python -c 'import __graft_entry__ as g; g.build()'` or "
            "`pyparrm_b200/csrc/build.sh`. pyparrm_b200 has no CPU fallback."
        )
    lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here = header/library mismatch
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.parrm_abi_version() != ABI_VERSION:
        raise ImportError(
            f"{LIB_NAME} has ABI version {lib.parrm_abi_version()}, expected {ABI_VERSION}; rebuild it."
        )
    return lib


lib = _load()


def last_error() -> str:
    msg = lib.parrm_last_error()
    return msg.decode("utf-8", "replace") if msg else ""


def check(status: int, what: str) -> None:
    """Raise if a C-ABI call did not return PARRM_OK."""
    if status != 0:
        raise RuntimeError(f"{what} failed (status {status}): {last_error()}")


def filter_last_kernel() -> str:
    """Name of the kernel this thread's last ``parrm_filter_apply*`` call enqueued."""
    name = lib.parrm_filter_last_kernel()
    return name.decode() if name else ""


def device_count() -> int:
    return int(lib.parrm_device_count())


def plan_filter(taps, dtype: int = F64, strategy: int = PLAN_AUTO):
    """Build a filter plan on the host; returns ``(plan_bytes, description)``.

    ``description`` is the decomposition the run-time specialised kernel evaluates: ``kind`` (0 gather,
    1 comb), ``stride``, ``windows`` (box lengths), ``boxes`` (one offset array per length),
    ``plus`` / ``minus`` single taps, ``centre`` and the modelled ``cost`` in loads per output.
    Pure host work: usable without a GPU.
    """
    import numpy as np

    taps = np.ascontiguousarray(taps, dtype=np.int32)
    nbytes = lib.parrm_filter_plan_bytes(taps.ctypes.data, int(taps.shape[0]))
    plan = np.zeros(nbytes, dtype=np.uint8)
    check(lib.parrm_filter_plan(taps.ctypes.data, int(taps.shape[0]), dtype, strategy,
                                plan.ctypes.data, nbytes), "parrm_filter_plan")
    info = np.zeros(16, dtype=np.int32)
    terms = np.zeros(256, dtype=np.int32)
    check(lib.parrm_filter_plan_info(plan.ctypes.data, info.ctypes.data, terms.ctypes.data, 256),
          "parrm_filter_plan_info")
    kind, stride, n_kinds, w0, w1, b0, b1, n_plus, n_minus, centre, cost = (int(v) for v in info[:11])
    cuts = np.cumsum([0, b0, b1, n_plus, n_minus])
    parts = [terms[cuts[i]:cuts[i + 1]].copy() for i in range(4)]
    desc = {
        "kind": kind, "stride": stride, "windows": [w0, w1][:n_kinds],
        "boxes": parts[:2][:n_kinds], "plus": parts[2], "minus": parts[3],
        "centre": centre, "cost": cost / 1000.0, "n_taps": int(info[11]),
    }
    return plan, desc

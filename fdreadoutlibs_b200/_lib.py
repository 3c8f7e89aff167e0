"""ctypes binding of libswtpg_b200.so (include/swtpg.h). The synthetic frame generator (include/swtpg_framegen.h) lives in
its own small library and module, fdreadoutlibs_b200/framegen.py.

The library is built in-tree by `make lib` / `__graft_entry__.build()`. There is deliberately no fallback: if the
shared object is missing, importing this module raises, and every compute call fails when no sm_100 GPU is present.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libswtpg_b200.so")

SWTPG_OK, SWTPG_ERR_INVALID_ARG, SWTPG_ERR_CUDA, SWTPG_ERR_BUSY, SWTPG_ERR_OVERFLOW, SWTPG_ERR_STATE, SWTPG_ERR_UNSUPPORTED = range(7)
FORMAT_WIBETH, FORMAT_WIB2 = 0, 1
ALGO_SIMPLE_THRESHOLD, ALGO_ABS_RS, ALGO_STANDARD_RS, ALGO_FIR_IQR = range(4)


class SwtpgConfig(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32),
        ("device", C.c_int32),
        ("format", C.c_int32),
        ("algorithm", C.c_int32),
        ("n_links", C.c_uint32),
        ("max_units", C.c_uint32),
        ("tp_capacity", C.c_uint32),
        ("n_slots", C.c_uint32),
        ("threshold", C.c_uint16),
        ("frugal_acc_limit", C.c_int16),
        ("rs_memory_factor", C.c_uint16),
        ("rs_scale_factor", C.c_uint16),
        ("fir_taps", C.c_int16 * 8),
        ("tap_exponent", C.c_uint8),
        ("reserved0", C.c_uint8 * 3),
        ("wib2_adc_offset", C.c_uint32),
        ("flags", C.c_uint32),
        ("dispatch_timeout_us", C.c_uint32),
    ]


MAX_LINK_CONFIGS = 16  # SWTPG_MAX_LINK_CONFIGS


class SwtpgLinkConfig(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32),
        ("algorithm", C.c_int32),
        ("threshold", C.c_uint16),
        ("frugal_acc_limit", C.c_int16),
        ("rs_memory_factor", C.c_uint16),
        ("rs_scale_factor", C.c_uint16),
        ("fir_taps", C.c_int16 * 8),
        ("tap_exponent", C.c_uint8),
        ("reserved0", C.c_uint8 * 3),
    ]


class SwtpgAdcStats(C.Structure):
    _fields_ = [
        ("samples", C.c_uint64),
        ("sum", C.c_uint64),
        ("sum_sq", C.c_uint64),
        ("min", C.c_uint16),
        ("max", C.c_uint16),
        ("reserved", C.c_uint32),
    ]


class SwtpgNoiseLags(C.Structure):
    _fields_ = [("segments", C.c_uint64), ("lag", C.c_uint64 * 33)]


class SwtpgCounters(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in (
        "units_processed", "samples_processed", "tps_emitted", "tps_dropped_overflow", "batches", "submit_busy",
        "h2d_bytes", "d2h_bytes", "units_zero_copy", "units_staged")]


# every symbol include/swtpg.h declares
EXPORTS = {
    "swtpg_abi_version": (C.c_uint32, []),
    "swtpg_status_string": (C.c_char_p, [C.c_int]),
    "swtpg_last_error": (C.c_char_p, [C.c_void_p]),
    "swtpg_device_available": (C.c_int, []),
    "swtpg_create": (C.c_int, [C.POINTER(SwtpgConfig), C.POINTER(C.c_void_p)]),
    "swtpg_destroy": (None, [C.c_void_p]),
    "swtpg_start": (C.c_int, [C.c_void_p]),
    "swtpg_stop": (C.c_int, [C.c_void_p]),
    "swtpg_set_rs_memory_factor": (C.c_int, [C.c_void_p, C.c_void_p]),
    "swtpg_set_link_rs_memory_factor": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p]),
    "swtpg_set_link_config": (C.c_int, [C.c_void_p, C.c_uint32, C.POINTER(SwtpgLinkConfig)]),
    "swtpg_set_link_thresholds": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p]),
    "swtpg_process_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]),
    "swtpg_process_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p]),
    "swtpg_fetch_tps": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]),
    "swtpg_last_kernel_ms": (C.c_double, [C.c_void_p]),
    "swtpg_process_host_debug": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_size_t,
                                           C.POINTER(C.c_size_t), C.c_void_p, C.c_void_p]),
    "swtpg_submit": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_size_t]),
    "swtpg_submit_wait": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p, C.c_size_t, C.c_uint64]),
    "swtpg_register_buffer": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "swtpg_unregister_buffer": (C.c_int, [C.c_void_p, C.c_void_p]),
    "swtpg_flush": (C.c_int, [C.c_void_p]),
    "swtpg_poll": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]),
    "swtpg_poll_wait": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t), C.c_uint64]),
    "swtpg_stream_status": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    "swtpg_stream_timing": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_uint64)]),
    "swtpg_sync": (C.c_int, [C.c_void_p]),
    "swtpg_dump_state": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p]),
    "swtpg_read_adc_stats": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_int]),
    "swtpg_read_noise_lags": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_int]),
    "swtpg_noise_power": (C.c_int, [C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]),
    "swtpg_read_channel_products": (C.c_int, [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_int]),
    "swtpg_channel_covariance": (C.c_int, [C.c_void_p, C.c_size_t, C.c_int, C.c_void_p, C.c_void_p]),
    "swtpg_get_counters": (C.c_int, [C.c_void_p, C.POINTER(SwtpgCounters)]),
    "swtpg_sort_stats": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "swtpg_alloc_pinned": (C.c_void_p, [C.c_size_t, C.c_int]),
    "swtpg_free_pinned": (None, [C.c_void_p]),
    "swtpg_sort_tps": (None, [C.c_void_p, C.c_size_t]),
    "swtpg_merge_sorted": (None, [C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.c_size_t, C.c_void_p]),
    "swtpg_firwin_int": (C.c_int, [C.c_int, C.c_double, C.c_int, C.c_void_p]),
}


def load() -> C.CDLL:
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `make lib` (or __graft_entry__.build()). "
            "fdreadoutlibs_b200 has no CPU fallback and will not run without its CUDA library.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in EXPORTS.items():
        fn = getattr(lib, name)  # AttributeError here = header and library out of sync
        fn.restype = res
        fn.argtypes = args
    return lib


lib = load()

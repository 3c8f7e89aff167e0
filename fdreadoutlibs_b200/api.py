"""Python face of the C ABI (include/swtpg.h), used by tests/, bench.py and examples.

`TPGenerator` is the batch/streaming generator for a set of links on one GPU; its methods map one-to-one onto the
C entry points, so the parity tests read like calls a C++ FrameProcessor would make.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import numpy as np

from . import frames as F
from ._lib import (ALGO_ABS_RS, ALGO_FIR_IQR, ALGO_SIMPLE_THRESHOLD, ALGO_STANDARD_RS, FORMAT_WIB2, FORMAT_WIBETH,
                   SWTPG_ERR_BUSY, SWTPG_ERR_OVERFLOW, SWTPG_OK, SwtpgConfig, SwtpgCounters, SwtpgLinkConfig, lib)

ALGORITHMS = {
    # tpg_algorithm strings of the reference (src/wibeth/WIBEthFrameProcessor.cpp:180-197)
    "SimpleThreshold": ALGO_SIMPLE_THRESHOLD,
    "AbsRS": ALGO_ABS_RS,
    "StandardRS": ALGO_STANDARD_RS,
    "FIR": ALGO_FIR_IQR,
}
FORMATS = {"wibeth": FORMAT_WIBETH, "wib2": FORMAT_WIB2}
FLAG_SORTED_TPS = 1  # SWTPG_FLAG_SORTED_TPS
FLAG_ADC_STATS = 2  # SWTPG_FLAG_ADC_STATS
FLAG_NOISE_SPECTRA = 8  # SWTPG_FLAG_NOISE_SPECTRA
FLAG_CHANNEL_COVARIANCE = 32  # SWTPG_FLAG_CHANNEL_COVARIANCE


class SwtpgError(RuntimeError):
    """`tps`: the records the failing call delivered all the same (poll on SWTPG_ERR_OVERFLOW), else None."""

    def __init__(self, status: int, detail: str, tps: Optional[np.ndarray] = None):
        self.status = status
        self.tps = tps
        super().__init__(f"{lib.swtpg_status_string(status).decode()} ({status}): {detail}")


class TPGAlgorithmInexistent(ValueError):
    """Mirrors the reference's ERS issue of the same name (include/fdreadoutlibs/FDReadoutIssues.hpp:27-31)."""


def device_available() -> bool:
    return bool(lib.swtpg_device_available())


def firwin_int(n: int = 7, cutoff: float = 0.1, multiplier: int = 64) -> np.ndarray:
    out = np.zeros(n, dtype=np.int16)
    lib.swtpg_firwin_int(n, cutoff, multiplier, out.ctypes.data)
    return out


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data


class TPGenerator:
    def __init__(self, n_links: int, max_units: int, *, fmt: str = "wibeth", algorithm: str = "SimpleThreshold", threshold: int = 60,
                 acc_limit: int = 10, rs_memory_factor: int = 8, rs_scale_factor: int = 5, fir_taps: Optional[Sequence[int]] = None,
                 tap_exponent: int = 6, tp_capacity: int = 0, n_slots: int = 0, device: int = 0, wib2_adc_offset: int = 0,
                 dispatch_timeout_us: int = 0, sorted_tps: bool = False, adc_stats: bool = False,
                 noise_spectra: bool = False, channel_covariance: bool = False):
        """sorted_tps: SWTPG_FLAG_SORTED_TPS — every batch's TP list comes back ordered by (time_start, link, channel), ordered on
        the device (include/swtpg.h). adc_stats: SWTPG_FLAG_ADC_STATS — per-channel ADC statistics of every batch, read by
        read_adc_stats(). noise_spectra: SWTPG_FLAG_NOISE_SPECTRA — per-channel noise lag sums of every batch, read by
        read_noise_lags() and turned into power spectra by noise_power(). channel_covariance: SWTPG_FLAG_CHANNEL_COVARIANCE — the
        sums of products of every pair of channels of each link, read by read_channel_products() and turned into covariance and
        correlation matrices by channel_covariance()."""
        if algorithm not in ALGORITHMS:
            raise TPGAlgorithmInexistent(algorithm)
        cfg = SwtpgConfig()
        cfg.struct_size = C.sizeof(SwtpgConfig)
        cfg.device = device
        cfg.format = FORMATS[fmt]
        cfg.algorithm = ALGORITHMS[algorithm]
        cfg.n_links = n_links
        cfg.max_units = max_units
        cfg.tp_capacity = tp_capacity
        cfg.n_slots = n_slots
        cfg.threshold = threshold
        cfg.frugal_acc_limit = acc_limit
        cfg.rs_memory_factor = rs_memory_factor
        cfg.rs_scale_factor = rs_scale_factor
        if fir_taps is not None:
            for i, t in enumerate(fir_taps):
                cfg.fir_taps[i] = int(t)
        cfg.tap_exponent = tap_exponent
        cfg.wib2_adc_offset = wib2_adc_offset
        cfg.dispatch_timeout_us = dispatch_timeout_us
        cfg.flags = ((FLAG_SORTED_TPS if sorted_tps else 0) | (FLAG_ADC_STATS if adc_stats else 0) | (FLAG_NOISE_SPECTRA if noise_spectra else 0)
                     | (FLAG_CHANNEL_COVARIANCE if channel_covariance else 0))
        self.cfg = cfg
        self.fmt = fmt
        self.n_links = n_links
        self.max_units = max_units
        self.unit_bytes = F.WIB2_SUPERCHUNK_BYTES if fmt == "wib2" else F.WIBETH_FRAME_BYTES
        self.channels = F.WIB2_CHANNELS if fmt == "wib2" else F.WIBETH_CHANNELS
        self.ticks = F.WIB2_SUPERCHUNK_FRAMES if fmt == "wib2" else F.WIBETH_TICKS
        self._h = C.c_void_p()
        st = lib.swtpg_create(C.byref(cfg), C.byref(self._h))
        if st != SWTPG_OK:
            raise SwtpgError(st, (lib.swtpg_last_error(None) or b"").decode())

    # -- lifecycle -------------------------------------------------------------------------------------------------------
    def _check(self, st: int, allow=()):
        if st != SWTPG_OK and st not in allow:
            raise SwtpgError(st, (lib.swtpg_last_error(self._h) or b"").decode())
        return st

    def start(self):
        self._check(lib.swtpg_start(self._h))
        return self

    def stop(self):
        self._check(lib.swtpg_stop(self._h))

    def close(self):
        if self._h:
            lib.swtpg_destroy(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_rs_memory_factor(self, by_link_channel: Optional[np.ndarray]):
        a = None if by_link_channel is None else np.ascontiguousarray(by_link_channel, dtype=np.uint16)
        if a is not None:
            assert a.size == self.n_links * self.channels
        self._check(lib.swtpg_set_rs_memory_factor(self._h, _ptr(a)))

    def set_link_rs_memory_factor(self, link: int, by_channel: np.ndarray):
        a = np.ascontiguousarray(by_channel, dtype=np.uint16)
        assert a.size == self.channels
        self._check(lib.swtpg_set_link_rs_memory_factor(self._h, link, a.ctypes.data))

    def set_link_config(self, link: int, *, algorithm: Optional[str] = None, threshold: Optional[int] = None,
                        acc_limit: Optional[int] = None, rs_memory_factor: Optional[int] = None, rs_scale_factor: Optional[int] = None,
                        fir_taps: Optional[Sequence[int]] = None, tap_exponent: Optional[int] = None, reset: bool = False):
        """swtpg_set_link_config: the TPG parameters of one link. A field left as None takes the handle's value; reset=True
        returns the link to the handle's configuration. Only while the handle is stopped; takes effect at the next start()."""
        if reset:
            self._check(lib.swtpg_set_link_config(self._h, link, None))
            return
        if algorithm is not None and algorithm not in ALGORITHMS:
            raise TPGAlgorithmInexistent(algorithm)
        h = self.cfg
        c = SwtpgLinkConfig()
        c.struct_size = C.sizeof(SwtpgLinkConfig)
        c.algorithm = h.algorithm if algorithm is None else ALGORITHMS[algorithm]
        c.threshold = h.threshold if threshold is None else threshold
        c.frugal_acc_limit = h.frugal_acc_limit if acc_limit is None else acc_limit
        c.rs_memory_factor = h.rs_memory_factor if rs_memory_factor is None else rs_memory_factor
        c.rs_scale_factor = h.rs_scale_factor if rs_scale_factor is None else rs_scale_factor
        taps = list(h.fir_taps) if fir_taps is None else list(fir_taps)
        for i in range(8):
            c.fir_taps[i] = int(taps[i]) if i < len(taps) else 0
        c.tap_exponent = h.tap_exponent if tap_exponent is None else tap_exponent
        self._check(lib.swtpg_set_link_config(self._h, link, C.byref(c)))

    def set_link_thresholds(self, link: int, by_channel: Optional[np.ndarray]):
        """swtpg_set_link_thresholds: per-channel hit thresholds of one link, by frame channel (0..32767 each); None returns the
        link to its configuration's threshold. SimpleThreshold and the WIBEth running sums only. Only while the handle is
        stopped; takes effect at the next start() and stays until reset."""
        a = None if by_channel is None else np.ascontiguousarray(by_channel, dtype=np.uint16)
        if a is not None:
            assert a.size == self.channels
        self._check(lib.swtpg_set_link_thresholds(self._h, link, _ptr(a)))

    # -- batch entry points ----------------------------------------------------------------------------------------------
    def _nunits(self, n_units):
        if n_units is None:
            return None
        a = np.ascontiguousarray(n_units, dtype=np.uint32)
        assert a.size == self.n_links
        return a

    def process_host(self, frames: np.ndarray, n_units=None, units_stride: Optional[int] = None, cap: int = 1 << 20, debug: bool = False,
                     out: Optional[np.ndarray] = None):
        """frames: uint8 [n_links, units_stride, unit_bytes]. Returns TPs (unsorted) and, if debug, (tps, pedestal, waveform).
        `out`: optional caller-owned TP_DTYPE array (pinned memory makes the D2H copy asynchronous-capable and avoids a
        staging copy); the result is then a view of its first n records instead of a fresh array."""
        frames = np.ascontiguousarray(frames, dtype=np.uint8)
        if units_stride is None:
            units_stride = frames.size // (self.n_links * self.unit_bytes)
        assert frames.size == self.n_links * units_stride * self.unit_bytes, "frames must be [n_links, units_stride, unit_bytes]"
        nu = self._nunits(n_units)
        if out is None:
            out = np.empty(cap, dtype=F.TP_DTYPE)
            own = True
        else:
            assert out.dtype == F.TP_DTYPE and out.flags["C_CONTIGUOUS"]
            cap, own = out.size, False
        n = C.c_size_t(0)
        if debug:
            shape = (self.n_links, units_stride, self.ticks, self.channels)
            ped = np.zeros(shape, dtype=np.int16)
            wav = np.zeros(shape, dtype=np.int16)
            st = lib.swtpg_process_host_debug(self._h, frames.ctypes.data, _ptr(nu), units_stride, out.ctypes.data, cap, C.byref(n),
                                              ped.ctypes.data, wav.ctypes.data)
            self._check(st)
            return out[: n.value].copy(), ped, wav
        st = lib.swtpg_process_host(self._h, frames.ctypes.data, _ptr(nu), units_stride, out.ctypes.data, cap, C.byref(n))
        self._check(st)
        return out[: n.value].copy() if own else out[: n.value]

    def process_device(self, d_frames_ptr: int, units_stride: int, n_units=None, stream: Optional[int] = None):
        """stream: a cudaStream_t handle (e.g. torch.cuda.current_stream().cuda_stream) or None for the handle's own
        stream. Handle value 0 (the legacy default stream, torch's default) is passed as cudaStreamLegacy."""
        nu = self._nunits(n_units)
        sp = None if stream is None else C.c_void_p(stream if stream != 0 else 1)
        self._check(lib.swtpg_process_device(self._h, C.c_void_p(d_frames_ptr), _ptr(nu), units_stride, sp))

    def fetch_tps(self, cap: int = 1 << 20) -> np.ndarray:
        out = np.zeros(cap, dtype=F.TP_DTYPE)
        n = C.c_size_t(0)
        self._check(lib.swtpg_fetch_tps(self._h, out.ctypes.data, cap, C.byref(n)))
        return out[: n.value].copy()

    def fetch_count(self) -> int:
        """Waits for the last device batch and returns its TP count without copying records."""
        n = C.c_size_t(0)
        self._check(lib.swtpg_fetch_tps(self._h, None, 0, C.byref(n)), allow=(SWTPG_ERR_OVERFLOW,))
        return n.value

    def last_kernel_ms(self) -> float:
        return float(lib.swtpg_last_kernel_ms(self._h))

    # -- streaming entry points --------------------------------------------------------------------------------------------
    def submit(self, link: int, unit: np.ndarray, wait_us: int = 0) -> bool:
        """One payload of one link. False = back-pressure (SWTPG_ERR_BUSY); wait_us > 0 sleeps up to that long for ring space."""
        unit = np.ascontiguousarray(unit, dtype=np.uint8)  # a contiguous uint8 view is passed by address (zero-copy ingest relies on it)
        if wait_us:
            st = lib.swtpg_submit_wait(self._h, link, unit.ctypes.data, unit.size, wait_us)
        else:
            st = lib.swtpg_submit(self._h, link, unit.ctypes.data, unit.size)
        return self._check(st, allow=(SWTPG_ERR_BUSY,)) == SWTPG_OK

    def register_buffer(self, buf: np.ndarray):
        """Zero-copy ingest: payloads submitted from inside `buf` (the latency buffer) are not copied by submit(); the copy
        engine reads them where they lie when their batch is dispatched. `buf` must stay alive and unmodified until sync()."""
        assert buf.flags["C_CONTIGUOUS"] and buf.dtype == np.uint8
        self._check(lib.swtpg_register_buffer(self._h, buf.ctypes.data, buf.nbytes))

    def unregister_buffer(self, buf: np.ndarray):
        self._check(lib.swtpg_unregister_buffer(self._h, buf.ctypes.data))

    def flush(self, busy_ok: bool = False) -> bool:
        """Dispatch everything submitted so far. SWTPG_ERR_BUSY — every batch holds un-polled TPs: poll, then flush again —
        raises unless busy_ok, in which case it is reported as False (drain() loops on it)."""
        return self._check(lib.swtpg_flush(self._h), allow=(SWTPG_ERR_BUSY,) if busy_ok else ()) == SWTPG_OK

    def sync(self):
        self._check(lib.swtpg_sync(self._h))

    def poll(self, cap: int = 1 << 16, wait_us: int = 0) -> np.ndarray:
        """SWTPG_ERR_OVERFLOW (a batch found more TPs than tp_capacity) raises SwtpgError with the records this call delivered
        in its `tps`: they are true records, and no later poll returns them."""
        out = np.zeros(cap, dtype=F.TP_DTYPE)
        n = C.c_size_t(0)
        if wait_us:
            st = lib.swtpg_poll_wait(self._h, out.ctypes.data, cap, C.byref(n), wait_us)
        else:
            st = lib.swtpg_poll(self._h, out.ctypes.data, cap, C.byref(n))
        if st == SWTPG_ERR_OVERFLOW:
            raise SwtpgError(st, (lib.swtpg_last_error(self._h) or b"").decode(), tps=out[: n.value].copy())
        self._check(st)
        return out[: n.value].copy()

    def drain(self) -> np.ndarray:
        """flush + sync + poll until nothing is left: every TP of everything submitted so far."""
        got = []
        while True:
            done = self.flush(busy_ok=True)
            self.sync()
            while True:
                part = self.poll()
                got.append(part)
                if part.size == 0 and self.stream_status()[2] == 0:
                    break
            if done and self.stream_status()[0] == 0:
                break
        return np.concatenate(got) if got else np.zeros(0, dtype=F.TP_DTYPE)

    def stream_status(self):
        """(units submitted but not dispatched, batches in flight, completed batches waiting for poll)"""
        a, b, c = C.c_uint64(0), C.c_uint32(0), C.c_uint32(0)
        self._check(lib.swtpg_stream_status(self._h, C.byref(a), C.byref(b), C.byref(c)))
        return a.value, b.value, c.value

    def stream_timing(self):
        """(device ms in the gather kernel, device ms in the TPG kernel, batches) of the streaming path since start()."""
        g, k, n = C.c_double(0), C.c_double(0), C.c_uint64(0)
        self._check(lib.swtpg_stream_timing(self._h, C.byref(g), C.byref(k), C.byref(n)))
        return g.value, k.value, n.value

    # -- parity / monitoring -------------------------------------------------------------------------------------------------
    def dump_state(self, link: int) -> np.ndarray:
        out = np.zeros(self.channels, dtype=F.STATE_DTYPE)
        self._check(lib.swtpg_dump_state(self._h, link, out.ctypes.data))
        return out

    def read_adc_stats(self, link0: int = 0, n_links: Optional[int] = None, reset: bool = False) -> np.ndarray:
        """swtpg_read_adc_stats: the current window of links [link0, link0 + n_links) (default: to the last link) as an
        (n_links, channels) ADC_STATS_DTYPE array, by frame channel. reset=True starts a new window of those links."""
        if n_links is None:
            n_links = max(0, self.n_links - link0)
        out = np.zeros((n_links, self.channels), dtype=F.ADC_STATS_DTYPE)
        self._check(lib.swtpg_read_adc_stats(self._h, link0, n_links, out.ctypes.data, 1 if reset else 0))
        return out

    def read_noise_lags(self, link0: int = 0, n_links: Optional[int] = None, reset: bool = False) -> np.ndarray:
        """swtpg_read_noise_lags: the current window of links [link0, link0 + n_links) (default: to the last link) as an
        (n_links, channels) NOISE_LAGS_DTYPE array, by frame channel. reset=True starts a new window of those links."""
        if n_links is None:
            n_links = max(0, self.n_links - link0)
        out = np.zeros((n_links, self.channels), dtype=F.NOISE_LAGS_DTYPE)
        self._check(lib.swtpg_read_noise_lags(self._h, link0, n_links, out.ctypes.data, 1 if reset else 0))
        return out

    def read_channel_products(self, link0: int = 0, n_links: Optional[int] = None, reset: bool = False) -> np.ndarray:
        """swtpg_read_channel_products: the current window of links [link0, link0 + n_links) (default: to the last link) as an
        (n_links, channel_products_words(fmt)) uint64 array in the header's layout (frames.unpack_channel_products splits a row).
        reset=True starts a new window of those links."""
        if n_links is None:
            n_links = max(0, self.n_links - link0)
        out = np.zeros((n_links, F.channel_products_words(self.fmt)), dtype=np.uint64)
        self._check(lib.swtpg_read_channel_products(self._h, link0, n_links, out.ctypes.data, 1 if reset else 0))
        return out

    def sort_stats(self) -> dict:
        """Device-side ordering (sorted_tps=True): ms of the last list, ms of all lists, lists ordered, lists the host finished."""
        a, b, n, f = C.c_double(0), C.c_double(0), C.c_uint64(0), C.c_uint64(0)
        self._check(lib.swtpg_sort_stats(self._h, C.byref(a), C.byref(b), C.byref(n), C.byref(f)))
        return {"last_ms": a.value, "total_ms": b.value, "lists": n.value, "finished_on_host": f.value}

    def counters(self) -> dict:
        c = SwtpgCounters()
        self._check(lib.swtpg_get_counters(self._h, C.byref(c)))
        return {n: int(getattr(c, n)) for n, _ in SwtpgCounters._fields_}


class PinnedBuffer:
    """Page-locked host memory from swtpg_alloc_pinned, viewed as a uint8 numpy array (`.array`). write_combined=True: the CPU
    should only write it (frames in); reads are very slow. Freed on close() / garbage collection."""

    def __init__(self, nbytes: int, write_combined: bool = False):
        self.ptr = lib.swtpg_alloc_pinned(nbytes, 1 if write_combined else 0)
        if not self.ptr:
            raise MemoryError(f"swtpg_alloc_pinned({nbytes}) failed")
        self.array = np.ctypeslib.as_array((C.c_uint8 * nbytes).from_address(self.ptr))

    def close(self):
        if getattr(self, "ptr", None):
            self.array = None
            lib.swtpg_free_pinned(self.ptr)
            self.ptr = None

    __del__ = close


def noise_power(lags: np.ndarray, fmt: str = "wibeth") -> np.ndarray:
    """swtpg_noise_power: the averaged periodogram of NOISE_LAGS_DTYPE entries of a `fmt` handle, shape lags.shape + (N/2 + 1,),
    in ADC counts^2 per bin (the mean over segments of |rfft(x)|^2 / N); bin k is at noise_frequencies(fmt)[k]. Entries without
    segments give zeros."""
    lags = np.ascontiguousarray(lags, dtype=F.NOISE_LAGS_DTYPE)
    out = np.zeros(lags.shape + (F.NOISE_SEGMENT_TICKS[fmt] // 2 + 1,), dtype=np.float64)
    st = lib.swtpg_noise_power(lags.ctypes.data, lags.size, FORMATS[fmt], out.ctypes.data)
    if st != SWTPG_OK:
        raise SwtpgError(st, "swtpg_noise_power")
    return out


def channel_covariance(products: np.ndarray, fmt: str = "wibeth"):
    """swtpg_channel_covariance of (n_links, channel_products_words(fmt)) rows of read_channel_products: (covariance,
    correlation), each (n_links, channels, channels) float64, by frame channel. Population covariance in ADC counts^2; the
    correlation is NaN in the row and column of a channel without variance, the covariance 0 there."""
    products = np.ascontiguousarray(products, dtype=np.uint64)
    if products.ndim != 2 or products.shape[1] != F.channel_products_words(fmt):
        raise ValueError(f"products must be (n_links, {F.channel_products_words(fmt)}) for {fmt}")
    c = F.WIB2_CHANNELS if fmt == "wib2" else F.WIBETH_CHANNELS
    cov = np.zeros((products.shape[0], c, c), dtype=np.float64)
    corr = np.zeros_like(cov)
    st = lib.swtpg_channel_covariance(products.ctypes.data, products.shape[0], FORMATS[fmt], cov.ctypes.data, corr.ctypes.data)
    if st != SWTPG_OK:
        raise SwtpgError(st, "swtpg_channel_covariance")
    return cov, corr


def noise_frequencies(fmt: str = "wibeth") -> np.ndarray:
    """Frequency in Hz of each bin of noise_power(.., fmt): k x 1.953125 MHz / N, k = 0 .. N/2."""
    n = F.NOISE_SEGMENT_TICKS[fmt]
    return np.arange(n // 2 + 1) * (F.SAMPLE_RATE_HZ / n)


def sort_tps(tps: np.ndarray) -> np.ndarray:
    """(time_start, link, channel) order via the library's host sort (swtpg_sort_tps)."""
    tps = np.ascontiguousarray(tps, dtype=F.TP_DTYPE).copy()
    lib.swtpg_sort_tps(tps.ctypes.data, tps.size)
    return tps


def merge_sorted(lists: Sequence[np.ndarray]) -> np.ndarray:
    """Host-side time-ordered k-way merge of per-GPU sorted TP lists (swtpg_merge_sorted)."""
    lists = [np.ascontiguousarray(x, dtype=F.TP_DTYPE) for x in lists]
    k = len(lists)
    out = np.zeros(sum(x.size for x in lists), dtype=F.TP_DTYPE)
    ptrs = (C.c_void_p * k)(*[x.ctypes.data for x in lists])
    ns = (C.c_size_t * k)(*[x.size for x in lists])
    lib.swtpg_merge_sorted(ptrs, ns, k, out.ctypes.data)
    return out


# -- synthetic frames (include/swtpg_framegen.h): re-exported from their own module / library ---------------------------------
from .framegen import GenParams, gen_params, gen_wib2_device, gen_wib2_host, gen_wibeth_device, gen_wibeth_host  # noqa: E402,F401

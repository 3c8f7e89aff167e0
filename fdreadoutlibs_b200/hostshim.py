"""ctypes face of libswtpg_host.so — the C++ frame-processor shim (fdreadoutlibs_b200/host/). Test harness only: a C++
application links the classes of swtpg_host.hpp directly."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
HOST_LIB_PATH = os.path.join(_HERE, "libswtpg_host.so")


class HostConf(C.Structure):
    _fields_ = [("device", C.c_int32), ("format", C.c_int32), ("n_links", C.c_uint32), ("superchunk_units", C.c_uint32),
                ("tpg_algorithm", C.c_char * 32), ("tpg_rs_memory_factor", C.c_float), ("tpg_rs_scale_factor", C.c_float),
                ("tpg_threshold", C.c_uint16), ("tpg_frugal_streaming_accumulator_limit", C.c_int16), ("tp_timeout", C.c_uint64),
                ("channel_mask", C.c_uint32 * 16), ("n_mask", C.c_uint32), ("crate_id", C.c_uint16), ("slot_id", C.c_uint16),
                ("first_link_id", C.c_uint16), ("enable_tpg", C.c_uint8), ("emulator_mode", C.c_uint8),
                ("correct_channel_lookup", C.c_uint8), ("reversed_map", C.c_uint8), ("enable_simple_threshold_on_collection", C.c_uint8),
                ("block_on_backpressure", C.c_uint8), ("count_only_sink", C.c_uint8), ("n_slots", C.c_uint8), ("sink_capacity", C.c_uint32)]


class HostLinkConf(C.Structure):
    _fields_ = [("tpg_algorithm", C.c_char * 32), ("tpg_rs_memory_factor", C.c_float), ("tpg_rs_scale_factor", C.c_float),
                ("tpg_threshold", C.c_uint16), ("tpg_frugal_streaming_accumulator_limit", C.c_int16),
                ("tpg_plane_threshold", C.c_int32 * 3)]


HOST_TP_DTYPE = np.dtype([("time_start", "<u8"), ("time_peak", "<u8"), ("time_over_threshold", "<u8"), ("channel", "<u4"),
                          ("adc_integral", "<u4"), ("adc_peak", "<u2"), ("detid", "<u2"), ("type", "<u4"), ("algorithm", "<u4"),
                          ("version", "<u2"), ("flag", "<u2")], align=True)


# ChannelAdcStats of swtpg_host.hpp
HOST_ADC_STATS_DTYPE = np.dtype([("offline_channel", "<u4"), ("samples", "<u8"), ("mean", "<f8"), ("rms", "<f8"), ("min", "<u2"),
                                 ("max", "<u2")], align=True)
assert HOST_ADC_STATS_DTYPE.itemsize == 40

# ChannelNoiseSpectrum of swtpg_host.hpp (WIB2 fills power[0..24])
HOST_NOISE_SPECTRUM_DTYPE = np.dtype([("offline_channel", "<u4"), ("segments", "<u8"), ("power", "<f8", (33,))], align=True)
assert HOST_NOISE_SPECTRUM_DTYPE.itemsize == 280


class HostInfo(C.Structure):
    _fields_ = [("num_seq_id_errors", C.c_uint64), ("min_seq_id_jump", C.c_int32), ("max_seq_id_jump", C.c_int32),
                ("num_ts_errors", C.c_uint64), ("rate_tp_hits", C.c_double), ("num_tps_sent", C.c_uint64),
                ("num_tps_suppressed_too_long", C.c_uint64), ("num_tps_send_failed", C.c_uint64), ("num_frames_dropped_busy", C.c_uint64),
                ("top_channels", C.c_uint32 * 10), ("top_channel_tps", C.c_uint32 * 10), ("n_top", C.c_uint32)]


class FeedStats(C.Structure):
    _fields_ = [("wall_s", C.c_double), ("feeder_cpu_s", C.c_double), ("payloads", C.c_uint64), ("late_bursts", C.c_uint64)]


class TpSetHdr(C.Structure):
    _fields_ = [("seqno", C.c_uint64), ("start_time", C.c_uint64), ("end_time", C.c_uint64), ("run_number", C.c_uint32),
                ("origin", C.c_uint32), ("type", C.c_uint32), ("n_objects", C.c_uint32)]


class TpHandlerInfo(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("num_tps_sent", "num_tpsets_sent", "num_tps_in_tpsets_send_failed", "num_tpsets_send_failed",
                                          "num_tps_suppressed_tardy", "num_heartbeats")]


EXPORTS = ["swtpg_host_tpsets_create", "swtpg_host_tpsets_destroy", "swtpg_host_tpsets_receive", "swtpg_host_tpsets_cycle",
           "swtpg_host_tpsets_cutoff", "swtpg_host_tpsets_count", "swtpg_host_tpsets_get", "swtpg_host_tpsets_info",
           "swtpg_host_push_parallel", "swtpg_host_push_feeders", "swtpg_host_tp_count", "swtpg_host_counters", "swtpg_host_stream_timing", "swtpg_host_last_error", "swtpg_host_create", "swtpg_host_destroy", "swtpg_host_start", "swtpg_host_stop", "swtpg_host_push",
           "swtpg_host_take_tps", "swtpg_host_get_info", "swtpg_host_error_count", "swtpg_host_misconfigurations",
           "swtpg_host_last_daq_time", "swtpg_host_register_channel_map", "swtpg_host_register_buffer", "swtpg_host_adc_stats",
           "swtpg_host_noise_spectra", "swtpg_host_channel_covariance"]

_lib = None


def host_lib():
    global _lib
    if _lib is None:
        lib = C.CDLL(HOST_LIB_PATH)
        lib.swtpg_host_last_error.restype = C.c_char_p
        lib.swtpg_host_create.restype = C.c_void_p
        lib.swtpg_host_create.argtypes = [C.POINTER(HostConf), C.POINTER(HostLinkConf), C.c_uint32]
        lib.swtpg_host_destroy.argtypes = [C.c_void_p]
        lib.swtpg_host_start.argtypes = [C.c_void_p]
        lib.swtpg_host_stop.argtypes = [C.c_void_p]
        lib.swtpg_host_push.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]
        lib.swtpg_host_push_parallel.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32]
        lib.swtpg_host_push_feeders.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_double, C.c_uint32,
                                                C.POINTER(FeedStats)]
        lib.swtpg_host_counters.argtypes = [C.c_void_p, C.c_void_p]
        lib.swtpg_host_stream_timing.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_uint64)]
        lib.swtpg_host_tp_count.restype = C.c_uint64
        lib.swtpg_host_tp_count.argtypes = [C.c_void_p]
        lib.swtpg_host_take_tps.restype = C.c_size_t
        lib.swtpg_host_take_tps.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p, C.c_size_t]
        lib.swtpg_host_get_info.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(HostInfo)]
        lib.swtpg_host_error_count.restype = C.c_uint64
        lib.swtpg_host_error_count.argtypes = [C.c_void_p, C.c_uint32, C.c_char_p]
        lib.swtpg_host_misconfigurations.restype = C.c_uint32
        lib.swtpg_host_misconfigurations.argtypes = [C.c_void_p, C.c_uint32]
        lib.swtpg_host_last_daq_time.restype = C.c_uint64
        lib.swtpg_host_last_daq_time.argtypes = [C.c_void_p, C.c_uint32]
        lib.swtpg_host_register_channel_map.argtypes = [C.c_void_p, C.c_uint32, C.c_void_p]
        lib.swtpg_host_register_buffer.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int]
        lib.swtpg_host_adc_stats.argtypes = [C.c_void_p, C.c_uint32, C.c_int, C.c_void_p, C.c_uint32]
        lib.swtpg_host_noise_spectra.argtypes = [C.c_void_p, C.c_uint32, C.c_int, C.c_void_p, C.c_uint32]
        lib.swtpg_host_channel_covariance.argtypes = [C.c_void_p, C.c_uint32, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                                      C.c_uint32]
        lib.swtpg_host_tpsets_create.restype = C.c_void_p
        lib.swtpg_host_tpsets_create.argtypes = [C.c_uint32, C.c_uint32, C.c_uint64, C.c_uint32, C.c_uint32]
        lib.swtpg_host_tpsets_destroy.argtypes = [C.c_void_p]
        lib.swtpg_host_tpsets_receive.restype = C.c_size_t
        lib.swtpg_host_tpsets_receive.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t]
        lib.swtpg_host_tpsets_cycle.argtypes = [C.c_void_p]
        lib.swtpg_host_tpsets_cutoff.restype = C.c_uint64
        lib.swtpg_host_tpsets_cutoff.argtypes = [C.c_void_p]
        lib.swtpg_host_tpsets_count.restype = C.c_size_t
        lib.swtpg_host_tpsets_count.argtypes = [C.c_void_p]
        lib.swtpg_host_tpsets_get.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(TpSetHdr), C.c_void_p, C.c_size_t]
        lib.swtpg_host_tpsets_info.argtypes = [C.c_void_p, C.POINTER(TpHandlerInfo)]
        _lib = lib
    return _lib


class HostError(RuntimeError):
    pass


class FrameProcessors:
    """n_links frame processors (WIBEthFrameProcessor / WIB2FrameProcessor) sharing one TpgEngine on one device."""

    def __init__(self, n_links: int, superchunk_units: int, fmt: str = "wibeth", algorithm: str = "SimpleThreshold", threshold: int = 60,
                 rs_memory_factor: float = 0.8, rs_scale_factor: float = 2.0, acc_limit: int = 10, tp_timeout: int = 10 ** 9, channel_mask=(),
                 crate_id: int = 1, slot_id: int = 0, first_link_id: int = 0, enable_tpg: bool = True, emulator_mode: bool = False,
                 correct_channel_lookup: bool = False, reversed_map: bool = False, collection_simple_threshold: bool = False,
                 sink_capacity: int = 0, block_on_backpressure: bool = True, device: int = 0, count_only_sink: bool = False,
                 n_slots: int = 4, link_confs=None, adc_stats: bool = False,
                 noise_spectra: bool = False, channel_covariance: bool = False):
        """link_confs: optional list of n_links dicts, each overriding algorithm, threshold, rs_memory_factor, rs_scale_factor
        and acc_limit for its link's conf(); the keys it leaves out take the arguments above. A dict may also set
        plane_threshold: three thresholds by plane (0 = collection), -1 = the link's threshold (tpg_plane_threshold).
        adc_stats: the engine's handle accumulates per-channel ADC statistics (SWTPG_FLAG_ADC_STATS), read by adc_stats().
        noise_spectra: it accumulates per-channel noise lags (SWTPG_FLAG_NOISE_SPECTRA), read as spectra by noise_spectra().
        channel_covariance: it accumulates the channel products of every link (SWTPG_FLAG_CHANNEL_COVARIANCE), read as covariance
        and correlation matrices by channel_covariance()."""
        c = HostConf()
        c.device, c.format, c.n_links, c.superchunk_units = device, 1 if fmt == "wib2" else 0, n_links, superchunk_units
        c.tpg_algorithm = algorithm.encode()
        c.tpg_threshold, c.tpg_rs_memory_factor, c.tpg_rs_scale_factor = threshold, rs_memory_factor, rs_scale_factor
        c.tpg_frugal_streaming_accumulator_limit, c.tp_timeout = acc_limit, tp_timeout
        for i, m in enumerate(channel_mask):
            c.channel_mask[i] = m
        c.n_mask = len(channel_mask)
        c.crate_id, c.slot_id, c.first_link_id = crate_id, slot_id, first_link_id
        c.enable_tpg, c.emulator_mode, c.correct_channel_lookup, c.reversed_map = enable_tpg, emulator_mode, correct_channel_lookup, reversed_map
        c.enable_simple_threshold_on_collection = collection_simple_threshold
        c.sink_capacity = sink_capacity
        c.block_on_backpressure = block_on_backpressure
        c.count_only_sink = count_only_sink
        c.n_slots = n_slots
        self.lib = host_lib()
        self.n_links = n_links
        links = None
        if link_confs is not None:
            assert len(link_confs) == n_links
            links = (HostLinkConf * n_links)()
            for l, lc in enumerate(link_confs):
                links[l].tpg_algorithm = lc.get("algorithm", algorithm).encode()
                links[l].tpg_threshold = lc.get("threshold", threshold)
                links[l].tpg_rs_memory_factor = lc.get("rs_memory_factor", rs_memory_factor)
                links[l].tpg_rs_scale_factor = lc.get("rs_scale_factor", rs_scale_factor)
                links[l].tpg_frugal_streaming_accumulator_limit = lc.get("acc_limit", acc_limit)
                for p, t in enumerate(lc.get("plane_threshold", (-1, -1, -1))):
                    links[l].tpg_plane_threshold[p] = t
        # SWTPG_FLAG_ADC_STATS, SWTPG_FLAG_NOISE_SPECTRA, SWTPG_FLAG_CHANNEL_COVARIANCE
        flags = (2 if adc_stats else 0) | (8 if noise_spectra else 0) | (32 if channel_covariance else 0)
        self.h = self.lib.swtpg_host_create(C.byref(c), links, flags)
        if not self.h:
            raise HostError(self.lib.swtpg_host_last_error().decode())

    def _check(self, rc):
        if rc != 0:
            raise HostError(self.lib.swtpg_host_last_error().decode())

    def start(self):
        self._check(self.lib.swtpg_host_start(self.h))

    def stop(self):
        self._check(self.lib.swtpg_host_stop(self.h))

    def push(self, link: int, payload: np.ndarray):
        """payload: writable uint8 array of one frame / superchunk (pre-process tasks may rewrite its header)."""
        assert payload.dtype == np.uint8 and payload.flags["C_CONTIGUOUS"] and payload.flags["WRITEABLE"]
        self._check(self.lib.swtpg_host_push(self.h, link, payload.ctypes.data))

    def push_parallel(self, payloads: np.ndarray):
        """payloads: writable uint8 [n_links, n_units, unit_bytes]; one C++ thread per link pushes its units concurrently."""
        assert payloads.dtype == np.uint8 and payloads.flags["C_CONTIGUOUS"] and payloads.flags["WRITEABLE"] and payloads.shape[0] == self.n_links
        self._check(self.lib.swtpg_host_push_parallel(self.h, payloads.ctypes.data, payloads.shape[1]))

    def push_feeders(self, payloads: np.ndarray, n_threads: int = 8, burst: int = 16, pace: float = 0.0, passes: int = 1) -> dict:
        """A few consumer threads, each serving many links round-robin (`burst` payloads per link and turn); pace > 0 = against
        the clock at that multiple of real time. Returns wall / feeder CPU seconds, payload count, bursts that ran late."""
        assert payloads.dtype == np.uint8 and payloads.flags["C_CONTIGUOUS"] and payloads.flags["WRITEABLE"] and payloads.shape[0] == self.n_links
        st = FeedStats()
        self._check(self.lib.swtpg_host_push_feeders(self.h, payloads.ctypes.data, payloads.shape[1], n_threads, burst, pace, passes, C.byref(st)))
        return {"wall_s": st.wall_s, "feeder_cpu_s": st.feeder_cpu_s, "payloads": int(st.payloads), "late_bursts": int(st.late_bursts)}

    def adc_stats(self, link: int, reset: bool = False) -> np.ndarray:
        """The processor's get_adc_stats: HOST_ADC_STATS_DTYPE entries by the offline channel its TPs carry (empty before its
        first frame). reset=True starts a new window of the link."""
        out = np.zeros(256, dtype=HOST_ADC_STATS_DTYPE)
        n = self.lib.swtpg_host_adc_stats(self.h, link, 1 if reset else 0, out.ctypes.data, out.size)
        if n < 0:
            raise HostError(self.lib.swtpg_host_last_error().decode())
        return out[:n].copy()

    def noise_spectra(self, link: int, reset: bool = False) -> np.ndarray:
        """The processor's get_noise_spectra: HOST_NOISE_SPECTRUM_DTYPE entries by the offline channel its TPs carry (empty
        before its first frame). reset=True starts a new window of the link."""
        out = np.zeros(256, dtype=HOST_NOISE_SPECTRUM_DTYPE)
        n = self.lib.swtpg_host_noise_spectra(self.h, link, 1 if reset else 0, out.ctypes.data, out.size)
        if n < 0:
            raise HostError(self.lib.swtpg_host_last_error().decode())
        return out[:n].copy()

    def channel_covariance(self, link: int, reset: bool = False) -> dict:
        """The processor's get_channel_covariance: samples, offline_channel (C,) uint32 of each row in frame-channel order, and the
        (C, C) covariance and correlation matrices (C = 0 before its first frame). reset=True starts a new window of the link."""
        samples = C.c_uint64(0)
        offline = np.zeros(256, dtype=np.uint32)
        cov = np.zeros((256, 256), dtype=np.float64)
        corr = np.zeros((256, 256), dtype=np.float64)
        n = self.lib.swtpg_host_channel_covariance(self.h, link, 1 if reset else 0, C.byref(samples), offline.ctypes.data, cov.ctypes.data,
                                                   corr.ctypes.data, offline.size)
        if n < 0:
            raise HostError(self.lib.swtpg_host_last_error().decode())
        shape = (n, n)
        return {"samples": samples.value, "offline_channel": offline[:n].copy(), "covariance": cov.reshape(-1)[:n * n].reshape(shape).copy(),
                "correlation": corr.reshape(-1)[:n * n].reshape(shape).copy()}

    def counters(self) -> dict:
        """swtpg_get_counters of the engine behind the processors."""
        from ._lib import SwtpgCounters

        c = SwtpgCounters()
        self._check(self.lib.swtpg_host_counters(self.h, C.byref(c)))
        return {n: int(getattr(c, n)) for n, _ in SwtpgCounters._fields_}

    def stream_timing(self) -> dict:
        """Device time the engine's batches spent in the gather kernel (host-link transfer) and in the TPG kernel."""
        g, k, n = C.c_double(0), C.c_double(0), C.c_uint64(0)
        self._check(self.lib.swtpg_host_stream_timing(self.h, C.byref(g), C.byref(k), C.byref(n)))
        return {"gather_ms": g.value, "kernel_ms": k.value, "batches": int(n.value)}

    def tp_count(self) -> int:
        """TPs accepted so far by count-only sinks (count_only_sink=True)."""
        return int(self.lib.swtpg_host_tp_count(self.h))

    def register_buffer(self, payloads: np.ndarray, on: bool = True):
        """Zero-copy ingest: declare `payloads` (the array later passed to push / push_parallel) as the latency buffer, so that
        find_hits hands the copy engine pointers instead of copying each frame. Unregister (on=False) before freeing it."""
        assert payloads.dtype == np.uint8 and payloads.flags["C_CONTIGUOUS"]
        self._check(self.lib.swtpg_host_register_buffer(self.h, payloads.ctypes.data, payloads.nbytes, 1 if on else 0))

    def take_tps(self, link: int, cap: int = 1 << 18) -> np.ndarray:
        out = np.zeros(cap, dtype=HOST_TP_DTYPE)
        n = self.lib.swtpg_host_take_tps(self.h, link, out.ctypes.data, cap)
        return out[:n].copy()

    def get_info(self, link: int) -> dict:
        i = HostInfo()
        self.lib.swtpg_host_get_info(self.h, link, C.byref(i))
        d = {n: getattr(i, n) for n, _ in HostInfo._fields_ if not n.startswith("top")}
        d["top"] = [(i.top_channels[k], i.top_channel_tps[k]) for k in range(i.n_top)]
        return d

    def error_count(self, link: int, name: str) -> int:
        return int(self.lib.swtpg_host_error_count(self.h, link, name.encode()))

    def misconfigurations(self, link: int) -> int:
        return int(self.lib.swtpg_host_misconfigurations(self.h, link))

    def last_daq_time(self, link: int) -> int:
        return int(self.lib.swtpg_host_last_daq_time(self.h, link))

    def register_channel_map(self, link: int) -> np.ndarray:
        out = np.zeros(64, dtype=np.uint32)
        self.lib.swtpg_host_register_channel_map(self.h, link, out.ctypes.data)
        return out

    def close(self):
        if self.h:
            self.lib.swtpg_host_destroy(self.h)
            self.h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


class TPSetHandler:
    """TPCTPRequestHandler (src/TPCTPRequestHandler.cpp): TPs in, time-ordered TPSets / heartbeats out."""

    def __init__(self, source_id=7, rate_hz=100, min_latency_ticks=100000, run_number=1, sink_capacity=0):
        self.lib = host_lib()
        self.h = self.lib.swtpg_host_tpsets_create(source_id, rate_hz, min_latency_ticks, run_number, sink_capacity)

    def receive(self, tps: np.ndarray) -> int:
        tps = np.ascontiguousarray(tps, dtype=HOST_TP_DTYPE)
        return int(self.lib.swtpg_host_tpsets_receive(self.h, tps.ctypes.data, tps.size))

    def cycle(self) -> bool:
        return bool(self.lib.swtpg_host_tpsets_cycle(self.h))

    def cutoff(self) -> int:
        return int(self.lib.swtpg_host_tpsets_cutoff(self.h))

    def sets(self):
        out = []
        for i in range(self.lib.swtpg_host_tpsets_count(self.h)):
            hdr = TpSetHdr()
            self.lib.swtpg_host_tpsets_get(self.h, i, C.byref(hdr), None, 0)
            objs = np.zeros(hdr.n_objects, dtype=HOST_TP_DTYPE)
            self.lib.swtpg_host_tpsets_get(self.h, i, C.byref(hdr), objs.ctypes.data, objs.size)
            out.append(({n: getattr(hdr, n) for n, _ in TpSetHdr._fields_}, objs))
        return out

    def info(self) -> dict:
        i = TpHandlerInfo()
        self.lib.swtpg_host_tpsets_info(self.h, C.byref(i))
        return {n: getattr(i, n) for n, _ in TpHandlerInfo._fields_}

    def close(self):
        if self.h:
            self.lib.swtpg_host_tpsets_destroy(self.h)
            self.h = None

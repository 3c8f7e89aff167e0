"""Host-side frame and record layouts (numpy): the byte formats on either side of the hot path.

WIBEth frame (7200 B) and WIB2 frame (472 B) bit layouts follow the reference's use of fddetdataformats
(`include/fdreadoutlibs/wibeth/tpg/FrameExpand.hpp:192-246`, `include/fdreadoutlibs/wib2/tpg/FrameExpand.hpp:193-209`,
`unittest/WIBEthFrameExpansion_test.cxx:105-150`): a tick row is 64 (resp. 256) little-endian 14-bit fields, channel c
at bits [14c, 14c+14). These helpers exist for tests, fixtures and examples; the product path never unpacks on the host.
"""
from __future__ import annotations

import numpy as np

WIBETH_FRAME_BYTES = 7200
WIBETH_HEADER_BYTES = 32
WIBETH_CHANNELS = 64
WIBETH_TICKS = 64
WIBETH_TS_PER_FRAME = 2048
WIB2_FRAME_BYTES = 472
WIB2_SUPERCHUNK_FRAMES = 12
WIB2_SUPERCHUNK_BYTES = WIB2_FRAME_BYTES * WIB2_SUPERCHUNK_FRAMES
WIB2_CHANNELS = 256
WIB2_ADC_OFFSET = 20
TS_PER_TICK = 32

# swtpg_tp of include/swtpg.h (32 bytes)
TP_DTYPE = np.dtype(
    [
        ("time_start", "<u8"),
        ("time_peak", "<u8"),
        ("time_over_threshold", "<u4"),
        ("adc_integral", "<u4"),
        ("adc_peak", "<u2"),
        ("channel", "<u2"),
        ("link", "<u4"),
    ],
    align=True,
)
assert TP_DTYPE.itemsize == 32

# swtpg_channel_state of include/swtpg.h
STATE_DTYPE = np.dtype(
    [
        ("pedestal", "<i2"), ("accum", "<i2"),
        ("quantile25", "<i2"), ("quantile75", "<i2"), ("accum25", "<i2"), ("accum75", "<i2"),
        ("rs", "<i2"), ("pedestal_rs", "<i2"), ("accum_rs", "<i2"),
        ("rs_memory_factor", "<u2"),
        ("prev_was_over", "<u2"), ("hit_charge", "<u2"), ("hit_tover", "<u2"),
        ("hit_peak_adc", "<u2"), ("hit_peak_time", "<u2"),
        ("initialized", "<u2"),
        ("prev_samp", "<i2", (8,)),
    ],
    align=True,
)
assert STATE_DTYPE.itemsize == 48

# swtpg_adc_stats of include/swtpg.h: one channel over one window of swtpg_read_adc_stats
ADC_STATS_DTYPE = np.dtype(
    [("samples", "<u8"), ("sum", "<u8"), ("sum_sq", "<u8"), ("min", "<u2"), ("max", "<u2"), ("reserved", "<u4")],
    align=True,
)
assert ADC_STATS_DTYPE.itemsize == 32

# swtpg_noise_lags of include/swtpg.h: one channel over one window of swtpg_read_noise_lags (WIB2 fills lag[0..24])
NOISE_LAGS_DTYPE = np.dtype([("segments", "<u8"), ("lag", "<u8", (33,))], align=True)
assert NOISE_LAGS_DTYPE.itemsize == 272
# SWTPG_*_NOISE_SEGMENT_TICKS: ticks per noise-spectrum segment (one WIBEth frame, four WIB2 superchunks)
NOISE_SEGMENT_TICKS = {"wibeth": 64, "wib2": 48}
SAMPLE_RATE_HZ = 62.5e6 / 32  # one ADC sample per channel every 32 ticks of the 62.5 MHz timing clock


def channel_products_words(fmt: str) -> int:
    """SWTPG_CHANNEL_PRODUCTS_WORDS: uint64 words per link of swtpg_read_channel_products (2145 WIBEth, 33153 WIB2)."""
    c = WIB2_CHANNELS if fmt == "wib2" else WIBETH_CHANNELS
    return 1 + c + c * (c + 1) // 2


def unpack_channel_products(words: np.ndarray, fmt: str):
    """One link's row of swtpg_read_channel_products -> (samples, sums (C,) uint64, products (C, C) uint64, full and symmetric)."""
    c = WIB2_CHANNELS if fmt == "wib2" else WIBETH_CHANNELS
    words = np.asarray(words, dtype=np.uint64)
    assert words.shape == (channel_products_words(fmt),), words.shape
    i, j = np.triu_indices(c)  # row-major upper triangle, i = 0 first: the header's order
    p = np.zeros((c, c), dtype=np.uint64)
    p[i, j] = words[1 + c:]
    p[j, i] = words[1 + c:]
    return int(words[0]), words[1:1 + c].copy(), p

# Lane l of AVX2 register r holds frame channel 16r + LANE_PERM[l] (unittest/WIBEthFrameExpansion_test.cxx:111,124).
LANE_PERM = np.array([0, 1, 2, 3, 4, 5, 6, 7, 15, 8, 9, 10, 11, 12, 13, 14], dtype=np.int64)


def position_to_channel(pos):
    """Register position (16r + lane) -> frame channel."""
    pos = np.asarray(pos)
    return (pos & ~15) | LANE_PERM[pos & 15]


def pack14(values: np.ndarray) -> np.ndarray:
    """Pack (..., n) integers (n multiple of 4) into (..., n*14/8) bytes, little-endian 14-bit fields."""
    v = np.asarray(values).astype(np.uint16) & 0x3FFF
    bits = ((v[..., None] >> np.arange(14, dtype=np.uint16)) & 1).astype(np.uint8)
    bits = bits.reshape(*v.shape[:-1], v.shape[-1] * 14)
    return np.packbits(bits, axis=-1, bitorder="little")


def unpack14(raw: np.ndarray, n: int) -> np.ndarray:
    """Inverse of pack14: (..., n*14/8) bytes -> (..., n) uint16."""
    bits = np.unpackbits(np.asarray(raw, dtype=np.uint8), axis=-1, bitorder="little")
    bits = bits.reshape(*raw.shape[:-1], n, 14).astype(np.uint16)
    return (bits << np.arange(14, dtype=np.uint16)).sum(axis=-1).astype(np.uint16)


def wibeth_header(timestamp: int, det_id=3, crate=1, slot=0, stream=0, seq=0) -> np.ndarray:
    """32-byte WIBEth header. Word 1 (bytes 8..15) is the timestamp (docs/README.md:81); the bit positions inside
    word 0 are restated from fddetdataformats (not in the reference tree, unpinned)."""
    w0 = (2 & 0x3F) | ((det_id & 0x3F) << 6) | ((crate & 0x3FF) << 12) | ((slot & 0xF) << 22) | ((stream & 0xFF) << 26)
    w0 |= ((seq & 0xFFF) << 40) | ((0x382 & 0xFFF) << 52)
    return np.array([w0, timestamp, 0, 0], dtype="<u8").view(np.uint8)


def pack_wibeth_frames(adc: np.ndarray, ts0: int, det_id=3, crate=1, slot=0, stream=0) -> np.ndarray:
    """adc: (F, 64 ticks, 64 channels) -> (F, 7200) uint8; frame f gets timestamp ts0 + 2048 f."""
    adc = np.asarray(adc)
    assert adc.ndim == 3 and adc.shape[1:] == (WIBETH_TICKS, WIBETH_CHANNELS), adc.shape
    out = np.zeros((adc.shape[0], WIBETH_FRAME_BYTES), dtype=np.uint8)
    for f in range(adc.shape[0]):
        out[f, :WIBETH_HEADER_BYTES] = wibeth_header(ts0 + WIBETH_TS_PER_FRAME * f, det_id, crate, slot, stream, seq=f)
    out[:, WIBETH_HEADER_BYTES:] = pack14(adc).reshape(adc.shape[0], -1)
    return out


def unpack_wibeth_frames(frames: np.ndarray):
    """(F, 7200) uint8 -> (adc (F, 64, 64) uint16, timestamps (F,) uint64)."""
    frames = np.asarray(frames, dtype=np.uint8).reshape(-1, WIBETH_FRAME_BYTES)
    ts = frames[:, 8:16].copy().view("<u8").reshape(-1)
    rows = frames[:, WIBETH_HEADER_BYTES:].reshape(-1, WIBETH_TICKS, 112)
    return unpack14(rows, WIBETH_CHANNELS), ts


def pack_wib2_superchunks(adc: np.ndarray, ts0: int, det_id=3, crate=1, slot=0, link=0, adc_offset=WIB2_ADC_OFFSET) -> np.ndarray:
    """adc: (T, 256) with T a multiple of 12 -> (T/12, 5664) uint8; frame t gets timestamp ts0 + 32 t."""
    adc = np.asarray(adc)
    assert adc.ndim == 2 and adc.shape[1] == WIB2_CHANNELS and adc.shape[0] % WIB2_SUPERCHUNK_FRAMES == 0
    n = adc.shape[0]
    out = np.zeros((n, WIB2_FRAME_BYTES), dtype=np.uint8)
    w0 = (4 & 0x3F) | ((det_id & 0x3F) << 6) | ((crate & 0x3FF) << 12) | ((slot & 0xF) << 22) | ((link & 0x3F) << 26)
    ts = ts0 + TS_PER_TICK * np.arange(n, dtype=np.uint64)
    hdr = np.zeros((n, 3), dtype="<u4")
    hdr[:, 0] = w0
    hdr[:, 1] = (ts & 0xFFFFFFFF).astype(np.uint32)
    hdr[:, 2] = (ts >> np.uint64(32)).astype(np.uint32)
    out[:, :12] = hdr.view(np.uint8).reshape(n, 12)
    out[:, adc_offset:adc_offset + 448] = pack14(adc)
    return out.reshape(n // WIB2_SUPERCHUNK_FRAMES, WIB2_SUPERCHUNK_BYTES)


def unpack_wib2_superchunks(sc: np.ndarray, adc_offset=WIB2_ADC_OFFSET):
    """(S, 5664) uint8 -> (adc (12 S, 256) uint16, timestamps (12 S,) uint64)."""
    fr = np.asarray(sc, dtype=np.uint8).reshape(-1, WIB2_FRAME_BYTES)
    w = fr[:, 4:12].copy().view("<u4").reshape(-1, 2).astype(np.uint64)
    ts = w[:, 0] | (w[:, 1] << np.uint64(32))
    return unpack14(fr[:, adc_offset:adc_offset + 448], WIB2_CHANNELS), ts


def sort_tps(tps: np.ndarray) -> np.ndarray:
    """Canonical order used by every comparison: (time_start, link, channel), then the remaining fields."""
    order = np.lexsort((tps["adc_integral"], tps["time_over_threshold"], tps["channel"], tps["link"], tps["time_start"]))
    return tps[order]

"""Per-channel noise spectra (SWTPG_FLAG_NOISE_SPECTRA, swtpg_read_noise_lags, swtpg_noise_power).

The device's lag sums are compared exactly with numpy int64 sums over the valid units of every batch: segments of N ticks (one
WIBEth frame, four WIB2 superchunks from a link's first valid unit of the batch, a remainder of 1-3 superchunks not counted), and
for each the circular lags sum_t x[t] x[(t + tau) mod N], tau = 0 .. N/2. swtpg_noise_power is compared with numpy's rfft."""
import ctypes as C
import os
import subprocess
import threading

import numpy as np
import pytest

import fdreadoutlibs_b200 as S
from fdreadoutlibs_b200 import _lib
from fdreadoutlibs_b200 import api as A
from fdreadoutlibs_b200 import frames as F
from fdreadoutlibs_b200 import hostshim as H
from util import (adc_of, all_wibeth_policies, channels, create_status, expected, expected_lags, lags_of, linear_map, ragged_batch, ragged_units,
                  run_device, sms)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- expected values --------------------------------------------------------------------------------------------------------------
def zeros(n_links, fmt):
    return np.zeros((n_links, channels(fmt)), dtype=F.NOISE_LAGS_DTYPE)


def add(a, b):
    out = a.copy()
    out["segments"] = a["segments"] + b["segments"]
    out["lag"] = a["lag"] + b["lag"]
    return out


def assert_lags(got, want, what):
    assert got.shape == want.shape, what
    for f in ("segments", "lag"):
        bad = np.argwhere((got[f] != want[f]).reshape(got.shape + (-1,)).any(axis=-1))
        if bad.size:
            l, c = bad[0]
            raise AssertionError(f"{what}: {len(bad)} (link, channel) differ in {f}; first: link {l} channel {c}: "
                                 f"got {got[l, c]} want {want[l, c]}")


# ---- CPU --------------------------------------------------------------------------------------------------------------------------
def test_noise_lags_layout_matches_the_header(tmp_path):
    """NOISE_LAGS_DTYPE and the ctypes mirror have the header's size and field offsets; the flag and segment lengths match."""
    src = tmp_path / "noise_lags_probe.c"
    src.write_text('#include "swtpg.h"\n#include <stddef.h>\n#include <stdio.h>\nint main(void) {\n'
                   '  printf("%zu %zu %zu %zu\\n", sizeof(swtpg_noise_lags), offsetof(swtpg_noise_lags, segments),'
                   ' offsetof(swtpg_noise_lags, lag), sizeof(((swtpg_noise_lags*)0)->lag));\n'
                   '  printf("%u %u %u\\n", SWTPG_FLAG_NOISE_SPECTRA, SWTPG_WIBETH_NOISE_SEGMENT_TICKS, SWTPG_WIB2_NOISE_SEGMENT_TICKS);\n'
                   '  return 0;\n}\n')
    exe = tmp_path / "noise_lags_probe"
    subprocess.run(["gcc", "-std=c11", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    size, off_seg, off_lag, lag_bytes, flag, n_eth, n_wib2 = (int(x) for x in subprocess.run([str(exe)], check=True, capture_output=True,
                                                                                            text=True).stdout.split())
    assert size == C.sizeof(_lib.SwtpgNoiseLags) == F.NOISE_LAGS_DTYPE.itemsize == 272
    assert off_seg == _lib.SwtpgNoiseLags.segments.offset == F.NOISE_LAGS_DTYPE.fields["segments"][1] == 0
    assert off_lag == _lib.SwtpgNoiseLags.lag.offset == F.NOISE_LAGS_DTYPE.fields["lag"][1] == 8
    assert lag_bytes == F.NOISE_LAGS_DTYPE.fields["lag"][0].itemsize == 33 * 8
    assert flag == A.FLAG_NOISE_SPECTRA == 8
    assert (n_eth, n_wib2) == (F.NOISE_SEGMENT_TICKS["wibeth"], F.NOISE_SEGMENT_TICKS["wib2"]) == (64, 48)


def periodogram(x):
    """Mean over segments of |rfft(x)|^2 / N: x (segments, N)."""
    return (np.abs(np.fft.rfft(x.astype(np.float64), axis=-1)) ** 2).mean(axis=0) / x.shape[-1]


@pytest.mark.parametrize("fmt", ["wibeth", "wib2"])
@pytest.mark.parametrize("pedestal,segments", [(900, 37), (16000, 37), (900, 1), (16000, 1), (None, 5)])
def test_noise_power_equals_the_rfft_periodogram(fmt, pedestal, segments):
    """swtpg_noise_power of lags built in numpy equals mean(|rfft(x)|^2) / N to 1e-9 of the total power: Gaussian noise with a
    line on bin 3 around pedestals near 900 and 16000, a single segment, and uniform random segments over the whole range."""
    n = F.NOISE_SEGMENT_TICKS[fmt]
    rng = np.random.default_rng([len(fmt), pedestal or 0, segments])
    if pedestal is None:
        x = rng.integers(0, 16384, (segments, 1, n))
    else:
        t = np.arange(n)
        x = np.clip(np.rint(rng.normal(pedestal, 25, (segments, 1, n)) + 40 * np.cos(2 * np.pi * 3 * t / n)), 0, 16383).astype(np.int64)
    lags = lags_of(fmt, x.transpose(0, 2, 1).reshape(-1, 1))
    got = S.noise_power(lags, fmt)[0]
    want = periodogram(x[:, 0, :])
    assert got.shape == (n // 2 + 1,)
    np.testing.assert_allclose(got, want, rtol=0, atol=1e-9 * want.sum())
    full = np.concatenate([got, got[1:-1][::-1]])  # the N bins of the full periodogram
    np.testing.assert_allclose(full.sum(), int(lags["lag"][0, 0]) / segments, rtol=1e-12)  # Parseval
    if pedestal is not None and segments > 1:
        assert np.argmax(got[1:]) + 1 == 3


def test_noise_power_shapes_and_empty_entries():
    lags = np.zeros((3, 4), dtype=F.NOISE_LAGS_DTYPE)
    assert S.noise_power(lags, "wibeth").shape == (3, 4, 33) and not S.noise_power(lags, "wibeth").any()
    assert S.noise_power(lags, "wib2").shape == (3, 4, 25)
    assert np.isclose(S.noise_frequencies("wibeth")[1], 30517.578125) and np.isclose(S.noise_frequencies("wib2")[1], 40690.104166666664)
    assert S.noise_frequencies("wibeth")[-1] == S.noise_frequencies("wib2")[-1] == 976562.5
    p = np.zeros(33)
    assert _lib.lib.swtpg_noise_power(lags.ctypes.data, 1, 7, p.ctypes.data) == _lib.SWTPG_ERR_UNSUPPORTED
    assert _lib.lib.swtpg_noise_power(None, 1, 0, p.ctypes.data) == _lib.SWTPG_ERR_INVALID_ARG


def test_read_noise_lags_without_handle():
    out = np.zeros(64, dtype=F.NOISE_LAGS_DTYPE)
    assert _lib.lib.swtpg_read_noise_lags(None, 0, 1, out.ctypes.data, 0) == _lib.SWTPG_ERR_INVALID_ARG


def test_create_accepts_the_statistics_flags_and_still_refuses_unknown_bits():
    """Flag bits 2 (ADC statistics) and 8 (noise spectra), alone and with the others, pass validation (no device here:
    SWTPG_ERR_CUDA; on a GPU: a handle); bit 4, bit 16 and above are still unknown."""
    known = (A.FLAG_ADC_STATS, A.FLAG_ADC_STATS | A.FLAG_SORTED_TPS, A.FLAG_NOISE_SPECTRA,
             A.FLAG_NOISE_SPECTRA | A.FLAG_ADC_STATS | A.FLAG_SORTED_TPS)
    for flags in known:
        assert create_status(flags=flags) in (_lib.SWTPG_OK, _lib.SWTPG_ERR_CUDA)
        assert create_status(fmt="wib2", flags=flags) in (_lib.SWTPG_OK, _lib.SWTPG_ERR_CUDA)
    for flags in (4, 4 | A.FLAG_NOISE_SPECTRA, 16, 16 | A.FLAG_NOISE_SPECTRA, 1 << 31):
        assert create_status(flags=flags) == _lib.SWTPG_ERR_INVALID_ARG


# ---- batch entry points -----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("fmt,adc_offset", [("wibeth", 0), ("wib2", 0), ("wib2", 24)])
def test_ragged_batches(fmt, adc_offset):
    """Three ragged batches (links of 0, 1 and units_stride units; WIB2 also every count 1..7, whose last 1-3 superchunks form no
    segment) through process_host and process_host_debug, with 0xFF past n_units and, for WIB2 at offset 24, before the ADC block."""
    n, stride = 24, 9
    specials = (0, 1, 2, 3, 4, 5, 6, 7, stride) if fmt == "wib2" else (0, 1, stride)
    gkw = dict(adc_offset=adc_offset) if fmt == "wib2" else {}
    off = adc_offset or F.WIB2_ADC_OFFSET
    want = zeros(n, fmt)
    with S.TPGenerator(n, stride, fmt=fmt, wib2_adc_offset=adc_offset, noise_spectra=True) as g:
        g.start()
        for k in range(3):
            nu = ragged_units(600 + k, n, stride, specials)
            frames = ragged_batch(fmt, 600 + k, n, stride, nu, **gkw)
            if fmt == "wib2" and adc_offset > 12:
                fr = frames.reshape(n, stride, F.WIB2_SUPERCHUNK_FRAMES, F.WIB2_FRAME_BYTES)
                fr[..., 12:adc_offset] = 0xFF
            want = add(want, expected_lags(fmt, frames, nu, off))
            g.process_host(frames, n_units=nu, debug=(k == 1))
        got = g.read_noise_lags()
    assert want["segments"].any()
    if fmt == "wib2":
        assert (want["lag"][..., 25:] == 0).all()
    assert_lags(got, want, f"{fmt} ragged batches")


@pytest.mark.gpu
def test_sinusoids_land_in_their_bins_and_lags_pass_32_bits():
    """Channel c carries a cosine on bin c % 32 + 1 over a pedestal with a little noise; channel 63 sits at 16383, so its lags
    pass 2^32 within one batch. Lags match numpy exactly, each line's power peaks in its bin, and the rail's power is all in
    bin 0."""
    n, stride = 2, 80
    rng = np.random.default_rng(610)
    t = np.arange(stride * 64).reshape(stride, 64, 1)
    k = (np.arange(64) % 32 + 1).reshape(1, 1, 64)
    adc = np.rint(900 + 300 * np.cos(2 * np.pi * k * t / 64) + rng.normal(0, 3, (n, stride, 64, 64)))
    adc = np.clip(adc, 0, 16383).astype(np.uint16)
    adc[..., 63] = 16383
    frames = np.stack([F.pack_wibeth_frames(adc[l], 1 << 40) for l in range(n)])
    with S.TPGenerator(n, stride, noise_spectra=True, tp_capacity=1 << 20) as g:  # the lines cross the threshold every period
        g.start()
        g.process_host(frames, cap=1 << 20)
        got = g.read_noise_lags()
    assert_lags(got, expected_lags("wibeth", frames), "sinusoids")
    rail = stride * 64 * 16383 ** 2
    assert rail > 2 ** 32 and (got["lag"][:, 63, :] == rail).all()
    power = S.noise_power(got)
    for c in range(63):
        assert (np.argmax(power[:, c, 1:], axis=-1) + 1).tolist() == [c % 32 + 1] * n, f"channel {c}"
    assert np.allclose(power[:, 63, 1:], 0, atol=1e-6 * power[:, 63, 0].max()) and np.allclose(power[:, 63, 0], 64 * 16383 ** 2)


@pytest.mark.gpu
def test_each_link_counted_once_with_several_configuration_groups():
    """A handle with every WIBEth policy (six configuration groups, six TPG launches per batch) counts each link once: its lags
    equal a uniform handle's and the numpy values."""
    policies = all_wibeth_policies()
    n, stride = 30, 8
    nus = [ragged_units(620 + k, n, stride, (0, 1, stride)) for k in range(2)]
    frames = [ragged_batch("wibeth", 620 + k, n, stride, nu) for k, nu in enumerate(nus)]
    got = []
    for mixed in (True, False):
        with S.TPGenerator(n, stride, noise_spectra=True) as g:
            if mixed:
                for l in range(n):
                    g.set_link_config(l, **policies[l % len(policies)])
            g.start()
            for f, nu in zip(frames, nus):
                g.process_host(f, n_units=nu)
            got.append(g.read_noise_lags())
    want = add(expected_lags("wibeth", frames[0], nus[0]), expected_lags("wibeth", frames[1], nus[1]))
    assert_lags(got[0], got[1], "mixed against uniform handle")
    assert_lags(got[0], want, "mixed handle")


# ---- windows ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_windows():
    n, stride = 12, 4
    frames = [ragged_batch("wib2", 630 + k, n, stride, np.full(n, stride)) for k in range(4)]
    per = [expected_lags("wib2", f) for f in frames]
    with S.TPGenerator(n, stride, fmt="wib2", noise_spectra=True) as g:
        assert_lags(g.read_noise_lags(), zeros(n, "wib2"), "before start")
        g.start()
        assert_lags(g.read_noise_lags(), zeros(n, "wib2"), "before the first batch")
        g.process_host(frames[0])
        assert_lags(g.read_noise_lags(), per[0], "one batch")
        g.process_host(frames[1])
        total = add(per[0], per[1])
        assert_lags(g.read_noise_lags(), total, "a read without reset accumulates")
        assert_lags(g.read_noise_lags(3, 5, reset=True), total[3:8], "a reset read of links 3..7")
        g.process_host(frames[2])
        w = g.read_noise_lags()
        assert_lags(w[3:8], per[2][3:8], "links 3..7 after their reset")
        keep = np.r_[0:3, 8:n]
        assert_lags(w[keep], add(total, per[2])[keep], "the other links keep their window")
        windows = [g.read_noise_lags(reset=True)]
        g.process_host(frames[3])
        windows.append(g.read_noise_lags(reset=True))
        assert_lags(windows[0], w, "first reset window")
        assert_lags(windows[1], per[3], "second reset window")
        g.process_host(frames[0])
        g.stop()
        assert_lags(g.read_noise_lags(), per[0], "readable after stop")
        g.start()
        assert_lags(g.read_noise_lags(), zeros(n, "wib2"), "start zeroes")
        with pytest.raises(S.SwtpgError) as e:
            g.read_noise_lags(10, 3)
        assert e.value.status == _lib.SWTPG_ERR_INVALID_ARG
        out = np.zeros(256, dtype=F.NOISE_LAGS_DTYPE)
        assert _lib.lib.swtpg_read_noise_lags(g._h, 0, 1, None, 0) == _lib.SWTPG_ERR_INVALID_ARG
        assert _lib.lib.swtpg_read_noise_lags(g._h, n, 0, out.ctypes.data, 0) == _lib.SWTPG_OK
        with pytest.raises(S.SwtpgError) as e:
            g.read_adc_stats()
        assert e.value.status == _lib.SWTPG_ERR_STATE
    with S.TPGenerator(n, stride, adc_stats=True) as g:
        g.start()
        with pytest.raises(S.SwtpgError) as e:
            g.read_noise_lags()
        assert e.value.status == _lib.SWTPG_ERR_STATE


@pytest.mark.gpu
def test_process_device_on_a_torch_stream():
    """A read straight after swtpg_process_device on a caller stream, with no host synchronisation, includes that batch; a reset
    read there ends the window exactly at that batch."""
    import torch

    n, stride = 240, 64
    host = S.gen_wibeth_host(S.gen_params(640, 0.3), n, stride)
    want = expected_lags("wibeth", host)
    s = torch.cuda.Stream()
    with S.TPGenerator(n, stride, noise_spectra=True) as g, torch.cuda.stream(s):
        g.start()
        buf = torch.from_numpy(host).pin_memory().to("cuda", non_blocking=True)  # on s
        for k in range(3):
            g.process_device(buf.data_ptr(), stride, stream=s.cuda_stream)
            assert_lags(g.read_noise_lags(reset=True), want, f"batch {k} read on the stream")
        g.process_device(buf.data_ptr(), stride, stream=s.cuda_stream)
        g.process_device(buf.data_ptr(), stride, stream=s.cuda_stream)
        got = g.read_noise_lags()
        g.sync()
    assert_lags(got, add(want, want), "two batches")


# ---- streaming path ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_streaming_path_with_a_concurrent_reader():
    """Frames of 24 WIBEth links, half zero-copy from a registered buffer and half staged, while a second thread reads with
    reset in a loop. After drain() and a final read the windows add up to numpy over every submitted frame (one segment each,
    so the batching of the streaming path does not change the sums)."""
    n, stride, n_units = 24, 8, 48
    units = S.gen_wibeth_host(S.gen_params(650, 0.3), n, n_units)
    latency = np.ascontiguousarray(units)
    staged = units.copy()
    windows, stop = [], threading.Event()
    with S.TPGenerator(n, stride, noise_spectra=True, dispatch_timeout_us=200) as g:
        g.register_buffer(latency.reshape(-1))
        g.start()

        def reader():
            while not stop.is_set():
                windows.append(g.read_noise_lags(reset=True))

        t = threading.Thread(target=reader)
        t.start()
        try:
            for u in range(n_units):
                for l in range(n):
                    assert g.submit(l, (latency if l < n // 2 else staged)[l, u], wait_us=1_000_000)
                g.poll()
        finally:
            stop.set()
            t.join()
        g.drain()
        windows.append(g.read_noise_lags())
        c = g.counters()
        g.stop()
    assert c["units_zero_copy"] > 0 and c["units_staged"] > 0
    assert len(windows) > 2
    total = windows[0]
    for w in windows[1:]:
        total = add(total, w)
    assert_lags(total, expected_lags("wibeth", units), "windows of the streaming path")


# ---- both flags -------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["wibeth", "wib2"])
def test_both_flags(fmt):
    """With both flags one kernel reads each batch once: its ADC statistics equal a statistics-only handle's, its lags a
    spectra-only handle's and numpy's; for WIBEth lag[0] is the sum of squares and segments x 64 the samples."""
    n, stride = 40, 11
    nus = [ragged_units(660 + k, n, stride, (0, 1, 2, 3, 5, stride)) for k in range(2)]
    frames = [ragged_batch(fmt, 660 + k, n, stride, nu) for k, nu in enumerate(nus)]
    got = {}
    for kw in (dict(adc_stats=True), dict(noise_spectra=True), dict(adc_stats=True, noise_spectra=True)):
        with S.TPGenerator(n, stride, fmt=fmt, **kw) as g:
            g.start()
            for f, nu in zip(frames, nus):
                g.process_host(f, n_units=nu)
            got[tuple(kw)] = (g.read_adc_stats() if kw.get("adc_stats") else None, g.read_noise_lags() if kw.get("noise_spectra") else None)
    stats, lags = got[("adc_stats", "noise_spectra")]
    assert (stats == got[("adc_stats",)][0]).all()
    assert (stats["samples"] == expected(fmt, frames[0], nus[0])["samples"] + expected(fmt, frames[1], nus[1])["samples"]).all()
    assert_lags(lags, got[("noise_spectra",)][1], "both flags against spectra only")
    assert_lags(lags, add(expected_lags(fmt, frames[0], nus[0]), expected_lags(fmt, frames[1], nus[1])), "both flags")
    if fmt == "wibeth":
        assert (lags["lag"][..., 0] == stats["sum_sq"]).all() and (lags["segments"] * 64 == stats["samples"]).all()


# ---- the flag changes nothing else ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_flag_changes_nothing_else_at_production_geometry():
    """A mixed SimpleThreshold / AbsRS / StandardRS handle at 20 warps per SM, ragged then full: TP lists, carried state and
    counters are bit-identical with the flag off and on."""
    per = 20 * sms() + 1
    n, stride = 3 * per, 64
    kinds = [dict(threshold=30), dict(algorithm="AbsRS", threshold=30), dict(algorithm="StandardRS", threshold=30, rs_memory_factor=6)]
    link_kw = {l: kinds[l % 3] for l in range(n)}
    nus = [ragged_units(670, n, stride, (0, 1, 16, 63, 64)), None]
    p = S.gen_params(670, 0.1)
    off = run_device("wibeth", n, stride, nus, p, link_kw=link_kw)
    on = run_device("wibeth", n, stride, nus, p, link_kw=link_kw, noise_spectra=True)
    for a, b in zip(off[0], on[0]):
        assert a.size > 10000 and np.array_equal(F.sort_tps(a), F.sort_tps(b))
    assert np.array_equal(off[1], on[1])
    assert off[2] == on[2]


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["wibeth", "wib2"])
def test_flag_changes_nothing_else_on_the_streaming_path(fmt):
    n, n_units = 16, 24
    gen = S.gen_wib2_host if fmt == "wib2" else S.gen_wibeth_host
    units = gen(S.gen_params(680, 0.3), n, n_units)
    got = []
    for on in (False, True):
        with S.TPGenerator(n, 8, fmt=fmt, noise_spectra=on) as g:
            g.start()
            parts = []
            for u in range(n_units):
                for l in range(n):
                    assert g.submit(l, units[l, u], wait_us=1_000_000)
                parts.append(g.poll())  # un-polled batches back-pressure the rings
            parts.append(g.drain())
            tps = F.sort_tps(np.concatenate(parts))
            got.append((tps, np.stack([g.dump_state(l) for l in range(n)])))
    assert got[0][0].size > 100 and np.array_equal(got[0][0], got[1][0])
    assert np.array_equal(got[0][1], got[1][1])


# ---- host shim --------------------------------------------------------------------------------------------------------------------
def reversed_map(crate, slot, stream, chan):
    return ((crate * 8 + slot) * 64 + stream) * 64 + (63 - chan)


@pytest.mark.gpu
@pytest.mark.parametrize("reversed_", [False, True])
@pytest.mark.parametrize("correct", [False, True])
def test_frame_processors_report_by_offline_channel(reversed_, correct):
    """get_noise_spectra of each WIBEth processor: one entry per frame channel under the offline channel its TPs carry (the H2
    switch correct_channel_lookup included), a masked channel too; segments and power as numpy computes them."""
    n_links, n_units, crate, slot, stream = 2, 16, 0, 1, 12
    m = reversed_map if reversed_ else linear_map
    units = S.gen_wibeth_host(S.gen_params(690, 0.3), n_links, n_units)
    masked = m(crate, slot, stream, 9)
    with H.FrameProcessors(n_links, 8, crate_id=crate, slot_id=slot, first_link_id=stream, emulator_mode=True, correct_channel_lookup=correct,
                           reversed_map=reversed_, channel_mask=(masked,), noise_spectra=True) as fp:
        assert fp.noise_spectra(0).size == 0  # no frame yet: no channel map
        fp.start()
        for u in range(n_units):
            for l in range(n_links):
                fp.push(l, units[l, u].copy())
        fp.stop()
        got = [fp.noise_spectra(l) for l in range(n_links)]
        maps = [fp.register_channel_map(l) for l in range(n_links)]
    for l in range(n_links):
        cr, sl, st = crate, slot, stream + l  # emulator mode writes the configured ids into every header
        offline = [m(cr, sl, st, c) if correct else int(maps[l][c]) for c in range(64)]
        a = adc_of("wibeth", units[l])
        g = got[l]
        assert g.size == 64 and g["offline_channel"].tolist() == offline
        assert (g["segments"] == n_units).all()
        want = np.stack([periodogram(a[:, c].reshape(n_units, 64)) for c in range(64)])
        assert (np.abs(g["power"] - want) <= 1e-9 * want.sum(axis=1, keepdims=True)).all()

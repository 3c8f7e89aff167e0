"""Per-channel ADC statistics (SWTPG_FLAG_ADC_STATS, swtpg_read_adc_stats).

The expected values are exact integer sums over the valid units of every batch, unpacked on the host by frames.py
(unpack_wibeth_frames / unpack_wib2_superchunks). The device must match them exactly for every link and channel: samples, sum,
sum of squares, minimum and maximum."""
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
from util import (adc_of, all_wibeth_policies, channels, combine, create_status, expected, linear_map, ragged_batch, ragged_units, run_device,
                  sms, stats_of)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- CPU --------------------------------------------------------------------------------------------------------------------------
def test_adc_stats_layout_matches_the_header(tmp_path):
    """ADC_STATS_DTYPE and the ctypes mirror have the header's size and field offsets (a C program prints them)."""
    fields = [n for n, _ in _lib.SwtpgAdcStats._fields_]
    src = tmp_path / "adc_stats_probe.c"
    src.write_text('#include "swtpg.h"\n#include <stddef.h>\n#include <stdio.h>\nint main(void) {\n'
                   '  printf("%zu\\n", sizeof(swtpg_adc_stats));\n'
                   + "".join(f'  printf("%zu\\n", offsetof(swtpg_adc_stats, {n}));\n' for n in fields)
                   + '  printf("%u\\n", SWTPG_FLAG_ADC_STATS);\n  return 0;\n}\n')
    exe = tmp_path / "adc_stats_probe"
    subprocess.run(["gcc", "-std=c11", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = [int(x) for x in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()]
    assert out[0] == C.sizeof(_lib.SwtpgAdcStats) == F.ADC_STATS_DTYPE.itemsize == 32
    assert out[1:-1] == [getattr(_lib.SwtpgAdcStats, n).offset for n in fields] == [F.ADC_STATS_DTYPE.fields[n][1] for n in fields]
    assert out[-1] == A.FLAG_ADC_STATS == 2


def test_read_adc_stats_without_handle():
    out = np.zeros(64, dtype=F.ADC_STATS_DTYPE)
    assert _lib.lib.swtpg_read_adc_stats(None, 0, 1, out.ctypes.data, 0) == _lib.SWTPG_ERR_INVALID_ARG


def test_create_accepts_the_flag_and_still_refuses_unknown_bits():
    """Flag bit 2 passes validation (no device here: SWTPG_ERR_CUDA; on a GPU: a handle); bit 4 is still unknown."""
    assert create_status(flags=A.FLAG_ADC_STATS) in (_lib.SWTPG_OK, _lib.SWTPG_ERR_CUDA)
    assert create_status(flags=A.FLAG_ADC_STATS | A.FLAG_SORTED_TPS) in (_lib.SWTPG_OK, _lib.SWTPG_ERR_CUDA)
    assert create_status(flags=4) == _lib.SWTPG_ERR_INVALID_ARG


# ---- expected values --------------------------------------------------------------------------------------------------------------
def zeros(n_links, fmt):
    return np.zeros((n_links, channels(fmt)), dtype=F.ADC_STATS_DTYPE)


def assert_stats(got, want, what):
    assert got.shape == want.shape, what
    for f in ("samples", "sum", "sum_sq", "min", "max"):
        bad = np.argwhere(got[f] != want[f])
        if bad.size:
            l, c = bad[0]
            raise AssertionError(f"{what}: {len(bad)} (link, channel) differ in {f}; first: link {l} channel {c}: "
                                 f"got {got[l, c]} want {want[l, c]}")
    assert not got["reserved"].any()


# ---- batch entry points -----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("fmt,adc_offset", [("wibeth", 0), ("wib2", 0), ("wib2", 24)])
def test_ragged_batches(fmt, adc_offset):
    """Three ragged batches (links of 0, 1 and units_stride units) through process_host and process_host_debug. WIB2 also runs
    with a non-default wib2_adc_offset and 0xFF in the bytes before the ADC block."""
    n, stride = 20, 8
    gkw = dict(adc_offset=adc_offset) if fmt == "wib2" else {}
    off = adc_offset or F.WIB2_ADC_OFFSET
    want = zeros(n, fmt)
    with S.TPGenerator(n, stride, fmt=fmt, wib2_adc_offset=adc_offset, adc_stats=True) as g:
        g.start()
        for k in range(3):
            nu = ragged_units(500 + k, n, stride, (0, 1, stride))
            frames = ragged_batch(fmt, 500 + k, n, stride, nu, **gkw)
            if fmt == "wib2" and adc_offset > 12:
                fr = frames.reshape(n, stride, F.WIB2_SUPERCHUNK_FRAMES, F.WIB2_FRAME_BYTES)
                fr[..., 12:adc_offset] = 0xFF
            want = combine(want, expected(fmt, frames, nu, off))
            g.process_host(frames, n_units=nu, debug=(k == 1))
        assert want["samples"].any() and (want["samples"] == 0).any()
        assert_stats(g.read_adc_stats(), want, f"{fmt} ragged batches")


@pytest.mark.gpu
def test_constant_noisy_and_saturated_channels():
    """Channels stuck at 0 and at 16383, a channel spanning the whole range, the rest Gaussian noise around a pedestal."""
    rng = np.random.default_rng(510)
    n, stride = 3, 6
    adc = np.clip(rng.normal(900, 25, (n, stride, 64, 64)), 0, 16383).astype(np.uint16)
    adc[..., 5] = 0
    adc[..., 6] = 16383
    adc[..., 7] = rng.integers(0, 16384, adc[..., 7].shape)
    frames = np.stack([F.pack_wibeth_frames(adc[l], 1 << 40) for l in range(n)])
    with S.TPGenerator(n, stride, adc_stats=True) as g:
        g.start()
        g.process_host(frames)
        got = g.read_adc_stats()
    assert_stats(got, expected("wibeth", frames), "constant / noisy channels")
    assert (got["min"][:, 5] == 0).all() and (got["max"][:, 5] == 0).all()
    assert (got["min"][:, 6] == 16383).all() and (got["max"][:, 6] == 16383).all()


@pytest.mark.gpu
def test_sums_of_squares_beyond_32_bits():
    """One batch of 4096 saturated frames (every ADC bit set): a channel's sum of squares passes 2^32 within every work item."""
    n, stride = 2, 4096
    frames = np.zeros((n, stride, F.WIBETH_FRAME_BYTES), dtype=np.uint8)
    frames[:, :, F.WIBETH_HEADER_BYTES:] = 0xFF
    with S.TPGenerator(n, stride, adc_stats=True) as g:
        g.start()
        g.process_host(frames)
        got = g.read_adc_stats()
    samples = stride * F.WIBETH_TICKS
    assert (got["samples"] == samples).all() and (got["sum"] == samples * 16383).all()
    assert (got["sum_sq"] == samples * 16383 ** 2).all()
    assert (got["min"] == 16383).all() and (got["max"] == 16383).all()


@pytest.mark.gpu
def test_each_link_counted_once_with_several_configuration_groups():
    """A handle with every WIBEth policy (six configuration groups, six launches per batch) counts each link once: its statistics
    equal a uniform handle's over the same frames, and the numpy values."""
    policies = all_wibeth_policies()
    n, stride = 30, 8
    batches = [(ragged_units(520 + k, n, stride, (0, 1, stride)), None) for k in range(2)]
    frames = [ragged_batch("wibeth", 520 + k, n, stride, nu) for k, (nu, _) in enumerate(batches)]
    got = []
    for mixed in (True, False):
        with S.TPGenerator(n, stride, adc_stats=True) as g:
            if mixed:
                for l in range(n):
                    g.set_link_config(l, **policies[l % len(policies)])
            g.start()
            for f, (nu, _) in zip(frames, batches):
                g.process_host(f, n_units=nu)
            got.append(g.read_adc_stats())
    want = combine(expected("wibeth", frames[0], batches[0][0]), expected("wibeth", frames[1], batches[1][0]))
    assert_stats(got[0], got[1], "mixed against uniform handle")
    assert_stats(got[0], want, "mixed handle")


# ---- windows ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_windows():
    n, stride = 12, 4
    frames = [ragged_batch("wibeth", 530 + k, n, stride, np.full(n, stride)) for k in range(4)]
    per = [expected("wibeth", f) for f in frames]
    with S.TPGenerator(n, stride, adc_stats=True) as g:
        assert_stats(g.read_adc_stats(), zeros(n, "wibeth"), "before start")
        g.start()
        assert_stats(g.read_adc_stats(), zeros(n, "wibeth"), "before the first batch")
        g.process_host(frames[0])
        assert_stats(g.read_adc_stats(), per[0], "one batch")
        g.process_host(frames[1])
        total = combine(per[0], per[1])
        assert_stats(g.read_adc_stats(), total, "a read without reset accumulates")
        assert_stats(g.read_adc_stats(3, 5, reset=True), total[3:8], "a reset read of links 3..7")
        g.process_host(frames[2])
        w = g.read_adc_stats()
        assert_stats(w[3:8], per[2][3:8], "links 3..7 after their reset")
        keep = np.r_[0:3, 8:n]
        assert_stats(w[keep], combine(total, per[2])[keep], "the other links keep their window")
        # reset windows add up to the total
        windows = [g.read_adc_stats(reset=True)]
        g.process_host(frames[3])
        windows.append(g.read_adc_stats(reset=True))
        assert_stats(windows[0], w, "first reset window")
        acc = combine(combine(combine(per[0], per[1]), per[2]), per[3])
        acc[3:8] = combine(per[2], per[3])[3:8]
        assert_stats(combine(windows[0], windows[1]), acc, "reset windows sum to the total")
        g.process_host(frames[0])
        g.stop()
        assert_stats(g.read_adc_stats(), per[0], "readable after stop")
        g.start()
        assert_stats(g.read_adc_stats(), zeros(n, "wibeth"), "start zeroes")
        with pytest.raises(S.SwtpgError) as e:
            g.read_adc_stats(10, 3)
        assert e.value.status == _lib.SWTPG_ERR_INVALID_ARG
        out = np.zeros(64, dtype=F.ADC_STATS_DTYPE)
        assert _lib.lib.swtpg_read_adc_stats(g._h, 0, 1, None, 0) == _lib.SWTPG_ERR_INVALID_ARG
        assert _lib.lib.swtpg_read_adc_stats(g._h, n, 0, out.ctypes.data, 0) == _lib.SWTPG_OK
    with S.TPGenerator(n, stride) as g:
        g.start()
        with pytest.raises(S.SwtpgError) as e:
            g.read_adc_stats()
        assert e.value.status == _lib.SWTPG_ERR_STATE


@pytest.mark.gpu
def test_process_device_on_a_torch_stream():
    """A read straight after swtpg_process_device on a caller stream, with no host synchronisation, includes that batch; a reset
    read there ends the window exactly at that batch."""
    import torch

    n, stride = 240, 64
    host = S.gen_wibeth_host(S.gen_params(540, 0.3), n, stride)
    want = expected("wibeth", host)
    s = torch.cuda.Stream()
    with S.TPGenerator(n, stride, adc_stats=True) as g, torch.cuda.stream(s):
        g.start()
        buf = torch.from_numpy(host).pin_memory().to("cuda", non_blocking=True)  # on s
        for k in range(3):
            g.process_device(buf.data_ptr(), stride, stream=s.cuda_stream)
            assert_stats(g.read_adc_stats(reset=True), want, f"batch {k} read on the stream")
        g.process_device(buf.data_ptr(), stride, stream=s.cuda_stream)
        g.process_device(buf.data_ptr(), stride, stream=s.cuda_stream)
        got = g.read_adc_stats()
        g.sync()
    twice = combine(want, want)
    assert_stats(got, twice, "two batches")


# ---- streaming path ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_streaming_path_with_a_concurrent_reader():
    """Units of 24 links, half zero-copy from a registered buffer and half staged, while a second thread reads with reset in a
    loop. TPs are polled as batches complete (un-polled batches back-pressure the rings). After drain() and a final read the
    windows add up to numpy over every submitted unit."""
    n, stride, n_units = 24, 8, 48
    units = S.gen_wibeth_host(S.gen_params(550, 0.3), n, n_units)
    latency = np.ascontiguousarray(units)  # registered: links 0..11 submit from here
    staged = units.copy()
    windows, stop = [], threading.Event()
    with S.TPGenerator(n, stride, adc_stats=True, dispatch_timeout_us=200) as g:
        g.register_buffer(latency.reshape(-1))
        g.start()

        def reader():
            while not stop.is_set():
                windows.append(g.read_adc_stats(reset=True))

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
        windows.append(g.read_adc_stats())
        c = g.counters()
        g.stop()
    assert c["units_zero_copy"] > 0 and c["units_staged"] > 0
    assert len(windows) > 2
    total = windows[0]
    for w in windows[1:]:
        total = combine(total, w)
    assert_stats(total, expected("wibeth", units), "windows of the streaming path")


# ---- full load --------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_full_load():
    """20 links per SM, 64 frames each, generated on the device; the statistics of a seeded sample of 64 links match numpy."""
    import torch

    n, stride = 20 * sms(), 64
    buf = torch.empty(n * stride * F.WIBETH_FRAME_BYTES, dtype=torch.uint8, device="cuda")
    try:
        S.gen_wibeth_device(S.gen_params(560, 0.1), buf.data_ptr(), n, stride)
        torch.cuda.synchronize()
        with S.TPGenerator(n, stride, adc_stats=True) as g:
            g.start()
            g.process_device(buf.data_ptr(), stride)
            got = g.read_adc_stats()
        links = np.sort(np.random.default_rng(560).choice(n, 64, replace=False))
        view = buf.view(n, stride, F.WIBETH_FRAME_BYTES)
        want = np.stack([stats_of(adc_of("wibeth", view[l].cpu().numpy())) for l in links])
    finally:
        del buf
        torch.cuda.empty_cache()
    assert (got["samples"] == stride * 64).all()
    assert_stats(got[links], want, "full load")


# ---- the flag changes nothing else ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_flag_changes_nothing_else_at_production_geometry():
    """A mixed SimpleThreshold / AbsRS / StandardRS handle at 20 warps per SM, ragged then full: TP lists, carried state and
    counters are bit-identical with the flag off and on."""
    per = 20 * sms() + 1
    n, stride = 3 * per, 64
    kinds = [dict(threshold=30), dict(algorithm="AbsRS", threshold=30), dict(algorithm="StandardRS", threshold=30, rs_memory_factor=6)]
    link_kw = {l: kinds[l % 3] for l in range(n)}
    nus = [ragged_units(570, n, stride, (0, 1, 16, 63, 64)), None]
    p = S.gen_params(570, 0.1)
    off = run_device("wibeth", n, stride, nus, p, link_kw=link_kw, adc_stats=False)
    on = run_device("wibeth", n, stride, nus, p, link_kw=link_kw, adc_stats=True)
    for a, b in zip(off[0], on[0]):
        assert a.size > 10000 and np.array_equal(F.sort_tps(a), F.sort_tps(b))
    assert np.array_equal(off[1], on[1])
    assert off[2] == on[2]


@pytest.mark.gpu
def test_flag_changes_nothing_else_on_the_streaming_path():
    n, n_units = 16, 24
    units = S.gen_wibeth_host(S.gen_params(580, 0.3), n, n_units)
    got = []
    for adc_stats in (False, True):
        with S.TPGenerator(n, 8, adc_stats=adc_stats) as g:
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
    """get_adc_stats of each WIBEth processor: one entry per frame channel under the offline channel its TPs carry (the H2 switch
    correct_channel_lookup included), a masked channel too; mean and RMS as numpy computes them."""
    n_links, n_units, crate, slot, stream = 2, 16, 0, 1, 12
    m = reversed_map if reversed_ else linear_map
    units = S.gen_wibeth_host(S.gen_params(590, 0.3), n_links, n_units)
    masked = m(crate, slot, stream, 9)
    with H.FrameProcessors(n_links, 8, crate_id=crate, slot_id=slot, first_link_id=stream, emulator_mode=True, correct_channel_lookup=correct,
                           reversed_map=reversed_, channel_mask=(masked,), adc_stats=True) as fp:
        assert fp.adc_stats(0).size == 0  # no frame yet: no channel map
        fp.start()
        for u in range(n_units):
            for l in range(n_links):
                fp.push(l, units[l, u].copy())
        fp.stop()
        got = [fp.adc_stats(l) for l in range(n_links)]
        maps = [fp.register_channel_map(l) for l in range(n_links)]
    for l in range(n_links):
        cr, sl, st = crate, slot, stream + l  # emulator mode writes the configured ids into every header
        offline = [m(cr, sl, st, c) if correct else int(maps[l][c]) for c in range(64)]
        assert [m(cr, sl, st, int(F.position_to_channel(p))) for p in range(64)] == maps[l].tolist()
        a = adc_of("wibeth", units[l]).astype(np.float64)
        g = got[l]
        assert g.size == 64 and g["offline_channel"].tolist() == offline
        assert (g["samples"] == a.shape[0]).all()
        np.testing.assert_allclose(g["mean"], a.mean(0), rtol=1e-12)
        np.testing.assert_allclose(g["rms"], a.std(0), rtol=1e-9)
        assert g["min"].tolist() == a.min(0).astype(int).tolist() and g["max"].tolist() == a.max(0).astype(int).tolist()

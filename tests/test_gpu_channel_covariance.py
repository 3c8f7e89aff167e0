"""Per-link channel covariance (SWTPG_FLAG_CHANNEL_COVARIANCE, swtpg_read_channel_products, swtpg_channel_covariance).

The device's words of every link are compared exactly with numpy over the valid units of every batch: the ticks counted, the sum of
every channel and the int64 matrix product x.T @ x of the unpacked ADC values (upper triangle, row-major). swtpg_channel_covariance
is compared with numpy.cov(bias=True) and numpy.corrcoef."""
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
from util import (adc_of, all_wibeth_policies, channels, create_status, expected, expected_products, linear_map, ragged_batch, ragged_units,
                  run_device, sms, words_of)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- expected values --------------------------------------------------------------------------------------------------------------
def zeros(n_links, fmt):
    return np.zeros((n_links, F.channel_products_words(fmt)), dtype=np.uint64)


def assert_products(got, want, fmt, what):
    assert got.shape == want.shape, f"{what}: shape {got.shape}, expected {want.shape}"
    bad = np.argwhere(got != want)
    if bad.size:
        l, k = (int(x) for x in bad[0])
        c = channels(fmt)
        if k == 0:
            where = "samples"
        elif k <= c:
            where = f"sum[{k - 1}]"
        else:
            i, j = np.triu_indices(c)
            where = f"products[{i[k - 1 - c]}][{j[k - 1 - c]}]"
        raise AssertionError(f"{what}: {len(bad)} words differ on {len(np.unique(bad[:, 0]))} links; first: link {l} {where}: "
                             f"got {got[l, k]} want {want[l, k]}")


def pack(fmt, adc, ts0=1 << 40):
    """adc (n_links, ticks, channels) -> frames (n_links, units, unit_bytes)."""
    if fmt == "wib2":
        return np.stack([F.pack_wib2_superchunks(a, ts0) for a in adc])
    return np.stack([F.pack_wibeth_frames(a.reshape(-1, F.WIBETH_TICKS, F.WIBETH_CHANNELS), ts0) for a in adc])


def ticks(fmt):
    return F.WIB2_SUPERCHUNK_FRAMES if fmt == "wib2" else F.WIBETH_TICKS


# ---- CPU --------------------------------------------------------------------------------------------------------------------------
def test_channel_products_layout_matches_the_header(tmp_path):
    """The flag, the word counts and the upper-triangle index of the header agree with Python and with numpy's triu order."""
    src = tmp_path / "products_probe.c"
    src.write_text('#include "swtpg.h"\n#include <stdio.h>\nint main(void) {\n'
                   '  printf("%u %u %u\\n", SWTPG_FLAG_CHANNEL_COVARIANCE, SWTPG_CHANNEL_PRODUCTS_WORDS(SWTPG_WIBETH_CHANNELS),'
                   ' SWTPG_CHANNEL_PRODUCTS_WORDS(SWTPG_WIB2_CHANNELS));\n'
                   '  return 0;\n}\n')
    exe = tmp_path / "products_probe"
    subprocess.run(["gcc", "-std=c11", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    flag, w_eth, w_wib2 = (int(x) for x in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split())
    assert flag == A.FLAG_CHANNEL_COVARIANCE == 32
    assert (w_eth, w_wib2) == (F.channel_products_words("wibeth"), F.channel_products_words("wib2")) == (2145, 33153)
    for fmt in ("wibeth", "wib2"):
        c = channels(fmt)
        i, j = np.triu_indices(c)
        assert (i * c - i * (i - 1) // 2 + (j - i) == np.arange(i.size)).all()  # k(i, j) of the header
        rng = np.random.default_rng(c)
        x = rng.integers(0, 16384, (37, c))
        samples, sums, p = F.unpack_channel_products(words_of(fmt, x), fmt)
        assert samples == 37 and (sums == x.sum(0)).all() and (p == x.T @ x).all() and (p == p.T).all()


@pytest.mark.parametrize("fmt", ["wibeth", "wib2"])
@pytest.mark.parametrize("pedestal", [900, 16000, None])
def test_channel_covariance_equals_numpy(fmt, pedestal):
    """Covariance against numpy.cov(bias=True) and correlation against numpy.corrcoef, on noise of sigma 3 with a shared
    component around pedestals of 900 and 16000 (where n P_ij and S_i S_j agree in their first 7 digits) and on uniform values."""
    c = channels(fmt)
    rng = np.random.default_rng([c, pedestal or 0])
    n = 3000
    if pedestal is None:
        x = rng.integers(0, 16384, (n, c))
    else:
        shared = rng.normal(0, 2, (n, 1)) * (np.arange(c) % 3 == 0)
        x = np.clip(np.rint(pedestal + rng.normal(0, 3, (n, c)) + shared), 0, 16383).astype(np.int64)
    words = np.stack([words_of(fmt, x), words_of(fmt, x[: n // 2])])
    cov, corr = S.channel_covariance(words, fmt)
    assert cov.shape == corr.shape == (2, c, c)
    for k, xs in enumerate((x, x[: n // 2])):
        want_cov = np.cov(xs.T, bias=True)
        want_corr = np.corrcoef(xs.T)
        np.testing.assert_allclose(cov[k], want_cov, rtol=0, atol=1e-9 * np.diag(want_cov).max())
        np.testing.assert_allclose(corr[k], want_corr, rtol=0, atol=1e-12)
        assert (cov[k] == cov[k].T).all() and (corr[k] == corr[k].T).all()
    if pedestal is not None:  # the shared component: channels 0, 3, 6, ... correlate
        assert corr[0, 0, 3] > 0.15 and abs(corr[0, 1, 2]) < 0.1


def test_channel_covariance_of_empty_and_constant_channels():
    """No samples: covariance 0, correlation NaN. A constant channel (dead, or on a rail): 0 and NaN in its row and column,
    the other channels unaffected. Either output may be NULL."""
    rng = np.random.default_rng(5)
    x = rng.integers(800, 1000, (500, 64))
    x[:, 7] = 0
    x[:, 40] = 16383
    words = np.stack([zeros(1, "wibeth")[0], words_of("wibeth", x)])
    cov, corr = S.channel_covariance(words)
    assert (cov[0] == 0).all() and np.isnan(corr[0]).all()
    for ch in (7, 40):
        assert (cov[1, ch] == 0).all() and (cov[1, :, ch] == 0).all()
        assert np.isnan(corr[1, ch]).all() and np.isnan(corr[1, :, ch]).all()
    live = np.setdiff1d(np.arange(64), [7, 40])
    np.testing.assert_allclose(corr[1][np.ix_(live, live)], np.corrcoef(x[:, live].T), rtol=0, atol=1e-12)
    only_cov = np.zeros((2, 64, 64))
    only_corr = np.zeros((2, 64, 64))
    assert _lib.lib.swtpg_channel_covariance(words.ctypes.data, 2, A.FORMAT_WIBETH, only_cov.ctypes.data, None) == _lib.SWTPG_OK
    assert _lib.lib.swtpg_channel_covariance(words.ctypes.data, 2, A.FORMAT_WIBETH, None, only_corr.ctypes.data) == _lib.SWTPG_OK
    assert _lib.lib.swtpg_channel_covariance(words.ctypes.data, 2, A.FORMAT_WIBETH, None, None) == _lib.SWTPG_OK
    assert (only_cov == cov).all() and np.array_equal(only_corr, corr, equal_nan=True)


def test_bad_arguments_are_refused():
    words = zeros(1, "wibeth")
    out = np.zeros((64, 64))
    assert _lib.lib.swtpg_channel_covariance(None, 1, A.FORMAT_WIBETH, out.ctypes.data, None) == _lib.SWTPG_ERR_INVALID_ARG
    assert _lib.lib.swtpg_channel_covariance(words.ctypes.data, 1, 7, out.ctypes.data, None) == _lib.SWTPG_ERR_UNSUPPORTED
    with pytest.raises(ValueError):
        S.channel_covariance(words, "wib2")  # a WIBEth row is too short for a WIB2 link
    with pytest.raises(ValueError):
        S.channel_covariance(words[0], "wibeth")
    assert _lib.lib.swtpg_read_channel_products(None, 0, 1, words.ctypes.data, 0) == _lib.SWTPG_ERR_INVALID_ARG


def test_create_accepts_the_covariance_flag_and_still_refuses_unknown_bits():
    """Bit 32 (channel covariance), alone and with each other flag, passes validation (no device here: SWTPG_ERR_CUDA; on a GPU:
    a handle); bits 4, 16 and 1 << 31 are still unknown, with it too."""
    cov = A.FLAG_CHANNEL_COVARIANCE
    for flags in (cov, cov | A.FLAG_SORTED_TPS, cov | A.FLAG_ADC_STATS, cov | A.FLAG_NOISE_SPECTRA,
                  cov | A.FLAG_SORTED_TPS | A.FLAG_ADC_STATS | A.FLAG_NOISE_SPECTRA):
        assert create_status(flags=flags) in (_lib.SWTPG_OK, _lib.SWTPG_ERR_CUDA)
        assert create_status(fmt="wib2", flags=flags) in (_lib.SWTPG_OK, _lib.SWTPG_ERR_CUDA)
    for flags in (4, 4 | cov, 16, 16 | cov, 1 << 31, (1 << 31) | cov):
        assert create_status(flags=flags) == _lib.SWTPG_ERR_INVALID_ARG


# ---- batch entry points -----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("fmt,adc_offset", [("wibeth", 0), ("wib2", 0), ("wib2", 24)])
def test_ragged_batches(fmt, adc_offset):
    """Three ragged batches (links of 0, 1 and units_stride units; WIB2 also every count 1..9 around its 8-unit slabs) through
    process_host and process_host_debug, with 0xFF past n_units and, for WIB2 at offset 24, before the ADC block."""
    n, stride = 24, 9
    specials = (0, 1, 2, 3, 4, 5, 6, 7, 8, stride) if fmt == "wib2" else (0, 1, stride)
    gkw = dict(adc_offset=adc_offset) if fmt == "wib2" else {}
    off = adc_offset or F.WIB2_ADC_OFFSET
    want = zeros(n, fmt)
    with S.TPGenerator(n, stride, fmt=fmt, wib2_adc_offset=adc_offset, channel_covariance=True) as g:
        g.start()
        for k in range(3):
            nu = ragged_units(700 + k, n, stride, specials)
            frames = ragged_batch(fmt, 700 + k, n, stride, nu, **gkw)
            if fmt == "wib2" and adc_offset > 12:
                fr = frames.reshape(n, stride, F.WIB2_SUPERCHUNK_FRAMES, F.WIB2_FRAME_BYTES)
                fr[..., 12:adc_offset] = 0xFF
            want += expected_products(fmt, frames, nu, off)
            g.process_host(frames, n_units=nu, debug=(k == 1))
        got = g.read_channel_products()
    assert (want[:, 0] > 0).any()
    assert_products(got, want, fmt, f"{fmt} ragged batches")


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["wibeth", "wib2"])
def test_values_on_both_sides_of_the_byte_split(fmt):
    """Every sample one of 0, 1, 255, 256, 257, 16127, 16128 and 16383 (high and low bytes at both ends), a few channels
    saturated at 16383 throughout: their products pass 2^32 within one work item. Two links, long enough that each is cut into
    several work items, and a third link with a ragged count."""
    c = channels(fmt)
    stride = 80 if fmt == "wibeth" else 72
    rng = np.random.default_rng(710)
    values = np.array([0, 1, 255, 256, 257, 16127, 16128, 16383])
    adc = values[rng.integers(0, values.size, (3, stride * ticks(fmt), c))]
    adc[:, :, [3, c - 1, c // 2]] = 16383
    adc[1, :, 5] = 0
    frames = pack(fmt, adc.astype(np.uint16))
    nu = np.array([stride, stride, stride - 13], dtype=np.uint32)
    with S.TPGenerator(3, stride, fmt=fmt, channel_covariance=True, tp_capacity=1 << 22) as g:
        g.start()
        g.process_host(frames, n_units=nu, cap=1 << 22)
        got = g.read_channel_products()
    want = expected_products(fmt, frames, nu)
    assert_products(got, want, fmt, f"{fmt} byte-split values")
    _, _, p = F.unpack_channel_products(got[0], fmt)
    assert int(p[3, 3]) == stride * ticks(fmt) * 16383 ** 2 > 2 ** 32


@pytest.mark.gpu
@pytest.mark.parametrize("fmt,group", [("wibeth", range(16, 32)), ("wib2", range(120, 136))])
def test_a_shared_signal_shows_as_a_correlation_block(fmt, group):
    """Independent noise of sigma 4 on a pedestal of 900 on every channel, plus one signal of sigma 12 shared by 16 channels (on
    WIB2 across the boundary of two 64-channel blocks): their correlations are near 1, every other one near 0."""
    c = channels(fmt)
    stride = 64 if fmt == "wibeth" else 256
    t = stride * ticks(fmt)
    rng = np.random.default_rng(720)
    adc = 900 + rng.normal(0, 4, (1, t, c))
    adc[0][:, list(group)] += rng.normal(0, 12, (t, 1))
    adc = np.clip(np.rint(adc), 0, 16383).astype(np.uint16)
    frames = pack(fmt, adc)
    with S.TPGenerator(1, stride, fmt=fmt, channel_covariance=True, threshold=200) as g:
        g.start()
        g.process_host(frames)
        got = g.read_channel_products()
    assert_products(got, expected_products(fmt, frames), fmt, "shared signal")
    cov, corr = S.channel_covariance(got, fmt)
    inside = np.zeros((c, c), dtype=bool)
    inside[np.ix_(list(group), list(group))] = True
    off_diag = ~np.eye(c, dtype=bool)
    assert corr[0][inside & off_diag].min() > 0.8
    assert np.abs(corr[0][~inside & off_diag]).max() < 0.15
    np.testing.assert_allclose(np.diag(cov[0]), adc[0].astype(np.float64).var(axis=0), rtol=1e-9)


@pytest.mark.gpu
def test_each_link_counted_once_with_several_configuration_groups():
    """A handle with every WIBEth policy (six configuration groups, six TPG launches per batch) counts each link once."""
    policies = all_wibeth_policies()
    n, stride = 30, 8
    nus = [ragged_units(730 + k, n, stride, (0, 1, stride)) for k in range(2)]
    frames = [ragged_batch("wibeth", 730 + k, n, stride, nu) for k, nu in enumerate(nus)]
    with S.TPGenerator(n, stride, channel_covariance=True) as g:
        for l in range(n):
            g.set_link_config(l, **policies[l % len(policies)])
        g.start()
        for f, nu in zip(frames, nus):
            g.process_host(f, n_units=nu)
        got = g.read_channel_products()
    want = expected_products("wibeth", frames[0], nus[0]) + expected_products("wibeth", frames[1], nus[1])
    assert_products(got, want, "wibeth", "six configuration groups")


# ---- windows ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_windows():
    n, stride = 12, 4
    fmt = "wib2"
    frames = [ragged_batch(fmt, 740 + k, n, stride, np.full(n, stride)) for k in range(4)]
    per = [expected_products(fmt, f) for f in frames]
    with S.TPGenerator(n, stride, fmt=fmt, channel_covariance=True) as g:
        assert_products(g.read_channel_products(), zeros(n, fmt), fmt, "before start")
        g.start()
        assert_products(g.read_channel_products(), zeros(n, fmt), fmt, "before the first batch")
        g.process_host(frames[0])
        assert_products(g.read_channel_products(), per[0], fmt, "one batch")
        g.process_host(frames[1])
        total = per[0] + per[1]
        assert_products(g.read_channel_products(), total, fmt, "a read without reset accumulates")
        assert_products(g.read_channel_products(3, 5, reset=True), total[3:8], fmt, "a reset read of links 3..7")
        g.process_host(frames[2])
        w = g.read_channel_products()
        assert_products(w[3:8], per[2][3:8], fmt, "links 3..7 after their reset")
        keep = np.r_[0:3, 8:n]
        assert_products(w[keep], (total + per[2])[keep], fmt, "the other links keep their window")
        windows = [g.read_channel_products(reset=True)]
        g.process_host(frames[3])
        windows.append(g.read_channel_products(reset=True))
        assert_products(windows[0], w, fmt, "first reset window")
        assert_products(windows[1], per[3], fmt, "second reset window")
        g.process_host(frames[0])
        g.stop()
        assert_products(g.read_channel_products(), per[0], fmt, "readable after stop")
        g.start()
        assert_products(g.read_channel_products(), zeros(n, fmt), fmt, "start zeroes")
        with pytest.raises(S.SwtpgError) as e:
            g.read_channel_products(10, 3)
        assert e.value.status == _lib.SWTPG_ERR_INVALID_ARG
        out = zeros(1, fmt)
        assert _lib.lib.swtpg_read_channel_products(g._h, 0, 1, None, 0) == _lib.SWTPG_ERR_INVALID_ARG
        assert _lib.lib.swtpg_read_channel_products(g._h, n, 0, out.ctypes.data, 0) == _lib.SWTPG_OK
        with pytest.raises(S.SwtpgError) as e:
            g.read_adc_stats()
        assert e.value.status == _lib.SWTPG_ERR_STATE
    with S.TPGenerator(n, stride, adc_stats=True, noise_spectra=True) as g:
        g.start()
        with pytest.raises(S.SwtpgError) as e:
            g.read_channel_products()
        assert e.value.status == _lib.SWTPG_ERR_STATE


@pytest.mark.gpu
def test_process_device_on_a_torch_stream():
    """A read straight after swtpg_process_device on a caller stream, with no host synchronisation, includes that batch; a reset
    read there ends the window exactly at that batch."""
    import torch

    n, stride = 240, 64
    host = S.gen_wibeth_host(S.gen_params(750, 0.3), n, stride)
    want = expected_products("wibeth", host)
    s = torch.cuda.Stream()
    with S.TPGenerator(n, stride, channel_covariance=True) as g, torch.cuda.stream(s):
        g.start()
        buf = torch.from_numpy(host).pin_memory().to("cuda", non_blocking=True)  # on s
        for k in range(3):
            g.process_device(buf.data_ptr(), stride, stream=s.cuda_stream)
            assert_products(g.read_channel_products(reset=True), want, "wibeth", f"batch {k} read on the stream")
        g.process_device(buf.data_ptr(), stride, stream=s.cuda_stream)
        g.process_device(buf.data_ptr(), stride, stream=s.cuda_stream)
        got = g.read_channel_products()
        g.sync()
    assert_products(got, want + want, "wibeth", "two batches")


# ---- streaming path ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_streaming_path_with_a_concurrent_reader():
    """Frames of 24 WIBEth links, half zero-copy from a registered buffer and half staged, while a second thread reads with
    reset in a loop. After drain() and a final read the windows add up to numpy over every submitted frame."""
    n, stride, n_units = 24, 8, 48
    units = S.gen_wibeth_host(S.gen_params(760, 0.3), n, n_units)
    latency = np.ascontiguousarray(units)
    staged = units.copy()
    windows, stop = [], threading.Event()
    with S.TPGenerator(n, stride, channel_covariance=True, dispatch_timeout_us=200) as g:
        g.register_buffer(latency.reshape(-1))
        g.start()

        def reader():
            while not stop.is_set():
                windows.append(g.read_channel_products(reset=True))

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
        windows.append(g.read_channel_products())
        c = g.counters()
        g.stop()
    assert c["units_zero_copy"] > 0 and c["units_staged"] > 0
    assert len(windows) > 2
    assert_products(np.sum(windows, axis=0, dtype=np.uint64), expected_products("wibeth", units), "wibeth", "windows of the streaming path")


# ---- all three statistics flags ---------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["wibeth", "wib2"])
def test_all_three_statistics_flags(fmt):
    """With the ADC statistics, the noise spectra and the covariance together, the first two read bit-identical to a handle
    without the covariance, and the products equal numpy's; samples, sums and the diagonal agree with the ADC statistics."""
    n, stride = 40, 11
    nus = [ragged_units(770 + k, n, stride, (0, 1, 2, 3, 5, 8, stride)) for k in range(2)]
    frames = [ragged_batch(fmt, 770 + k, n, stride, nu) for k, nu in enumerate(nus)]
    got = {}
    for cov in (False, True):
        with S.TPGenerator(n, stride, fmt=fmt, adc_stats=True, noise_spectra=True, channel_covariance=cov) as g:
            g.start()
            for f, nu in zip(frames, nus):
                g.process_host(f, n_units=nu)
            got[cov] = (g.read_adc_stats(), g.read_noise_lags(), g.read_channel_products() if cov else None)
    assert (got[False][0] == got[True][0]).all()
    assert (got[False][1] == got[True][1]).all()
    products = got[True][2]
    assert_products(products, expected_products(fmt, frames[0], nus[0]) + expected_products(fmt, frames[1], nus[1]), fmt, "three flags")
    stats = got[True][0]
    assert (stats["samples"] == expected(fmt, frames[0], nus[0])["samples"] + expected(fmt, frames[1], nus[1])["samples"]).all()
    for l in range(n):
        samples, sums, p = F.unpack_channel_products(products[l], fmt)
        assert (stats["samples"][l] == samples).all() and (stats["sum"][l] == sums).all() and (stats["sum_sq"][l] == np.diag(p)).all()


# ---- the flag changes nothing else ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_flag_changes_nothing_else_at_production_geometry():
    """A mixed SimpleThreshold / AbsRS / StandardRS handle at 20 warps per SM, ragged then full: TP lists, carried state and
    counters are bit-identical with the flag off and on."""
    per = 20 * sms() + 1
    n, stride = 3 * per, 64
    kinds = [dict(threshold=30), dict(algorithm="AbsRS", threshold=30), dict(algorithm="StandardRS", threshold=30, rs_memory_factor=6)]
    link_kw = {l: kinds[l % 3] for l in range(n)}
    nus = [ragged_units(780, n, stride, (0, 1, 16, 63, 64)), None]
    p = S.gen_params(780, 0.1)
    off = run_device("wibeth", n, stride, nus, p, link_kw=link_kw)
    on = run_device("wibeth", n, stride, nus, p, link_kw=link_kw, channel_covariance=True)
    for a, b in zip(off[0], on[0]):
        assert a.size > 10000 and np.array_equal(F.sort_tps(a), F.sort_tps(b))
    assert np.array_equal(off[1], on[1])
    assert off[2] == on[2]


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["wibeth", "wib2"])
def test_flag_changes_nothing_else_on_the_streaming_path(fmt):
    n, n_units = 16, 24
    gen = S.gen_wib2_host if fmt == "wib2" else S.gen_wibeth_host
    units = gen(S.gen_params(790, 0.3), n, n_units)
    got = []
    for on in (False, True):
        with S.TPGenerator(n, 8, fmt=fmt, channel_covariance=on) as g:
            g.start()
            parts = []
            for u in range(n_units):
                for l in range(n):
                    assert g.submit(l, units[l, u], wait_us=1_000_000)
                parts.append(g.poll())  # un-polled batches back-pressure the rings
            parts.append(g.drain())
            tps = F.sort_tps(np.concatenate(parts))
            got.append((tps, np.stack([g.dump_state(l) for l in range(n)]), g.read_channel_products() if on else None))
    assert got[0][0].size > 100 and np.array_equal(got[0][0], got[1][0])
    assert np.array_equal(got[0][1], got[1][1])
    assert_products(got[1][2], expected_products(fmt, units), fmt, "streaming path")


# ---- host shim --------------------------------------------------------------------------------------------------------------------
def reversed_map(crate, slot, stream, chan):
    return ((crate * 8 + slot) * 64 + stream) * 64 + (63 - chan)


@pytest.mark.gpu
@pytest.mark.parametrize("reversed_", [False, True])
def test_frame_processors_report_by_offline_channel(reversed_):
    """channel_covariance of each WIBEth processor: rows in frame-channel order under the offline channel its TPs carry, a
    masked channel too; samples, covariance and correlation as numpy computes them."""
    n_links, n_units, crate, slot, stream = 2, 16, 0, 1, 12
    m = reversed_map if reversed_ else linear_map
    units = S.gen_wibeth_host(S.gen_params(800, 0.3), n_links, n_units)
    masked = m(crate, slot, stream, 9)
    with H.FrameProcessors(n_links, 8, crate_id=crate, slot_id=slot, first_link_id=stream, emulator_mode=True, correct_channel_lookup=True,
                           reversed_map=reversed_, channel_mask=(masked,), channel_covariance=True) as fp:
        assert fp.channel_covariance(0)["offline_channel"].size == 0  # no frame yet: no channel map
        fp.start()
        for u in range(n_units):
            for l in range(n_links):
                fp.push(l, units[l, u].copy())
        fp.stop()
        got = [fp.channel_covariance(l) for l in range(n_links)]
        again = fp.channel_covariance(0, reset=True)
        empty = fp.channel_covariance(0)
    for l in range(n_links):
        a = adc_of("wibeth", units[l]).astype(np.float64)
        g = got[l]
        assert g["offline_channel"].tolist() == [m(crate, slot, stream + l, c) for c in range(64)]
        assert g["samples"] == n_units * 64
        np.testing.assert_allclose(g["covariance"], np.cov(a.T, bias=True), rtol=0, atol=1e-9 * a.var(axis=0).max())
        np.testing.assert_allclose(g["correlation"], np.corrcoef(a.T), rtol=0, atol=1e-12)
    assert again["samples"] == n_units * 64 and empty["samples"] == 0 and np.isnan(empty["correlation"]).all()

"""GPU (B200): parity of the CUDA path — always called through the C ABI (include/swtpg.h) — against the CPU oracle and the
reference-generated golden vectors. Bit-exact: TP field tuples, carried state, pedestal and waveform dumps."""
import os
import subprocess
import sys
import time

import numpy as np
import pytest

import cases
import fdreadoutlibs_b200 as S
from fdreadoutlibs_b200 import frames as F
from oracle import binding as B
from util import assert_same_as_reference, assert_same_state, assert_same_tps, dump_states, oracle_config

pytestmark = pytest.mark.gpu

WIBETH_CASES = sorted(n for n, c in cases.GOLDEN_CASES.items() if c["fmt"] == "wibeth" and c["flavour"] == 0)
WIB2_CASES = sorted(n for n, c in cases.GOLDEN_CASES.items() if c["fmt"] == "wib2" and c["flavour"] == 0)


def run_gpu(case, units, max_units=None, **kw):
    n_links, n_units = units.shape[0], units.shape[1]
    with S.TPGenerator(n_links, max_units or n_units, fmt=case["fmt"], algorithm=case["algorithm"], threshold=case["threshold"],
                       acc_limit=case.get("acc_limit", 10), rs_memory_factor=case.get("rs_memory_factor", 8),
                       rs_scale_factor=case.get("rs_scale_factor", 5), **kw) as g:
        g.start()
        step = max_units or n_units
        parts = [g.process_host(np.ascontiguousarray(units[:, u:u + step])) for u in range(0, n_units, step)]
        ped = np.stack([g.dump_state(l)["pedestal"] for l in range(n_links)])
        return np.concatenate(parts), ped


@pytest.mark.parametrize("name", WIBETH_CASES + WIB2_CASES)
def test_golden_cases(name, golden):
    """Same inputs as tests/golden/make_golden.py fed the reference with: TPs and final pedestals must be identical."""
    case = cases.GOLDEN_CASES[name]
    units = cases.make_input(case)
    tps, ped = run_gpu(case, units)
    assert_same_tps(tps, golden[name + "__tps"], name)
    assert (ped == golden[name + "__pedestal"]).all()


NAIVE_CASES = sorted(n for n, c in cases.GOLDEN_CASES.items() if c["flavour"] == 1)


@pytest.mark.parametrize("name", NAIVE_CASES)
def test_naive_golden_cases_where_defined(name, golden):
    """north_star: bit-exact against the reference's naive AND AVX2 processors. The CUDA path follows the AVX2 code (the
    production one); the scalar code agrees with it wherever SURVEY H3-H7 say the two are defined alike — accumulator limit 10,
    charge below 32768, FIR threshold 5 with sigma below its clamp — after mapping the naive record's register position to
    the frame channel. These are the reference's own NAIVE outputs (tests/golden/make_golden.py, ref_impl of the case).
    The one documented divergence, charge overflow (H3: AVX2 wraps mod 2^16, the scalar code saturates), is asserted as such."""
    case = cases.GOLDEN_CASES[name]
    tps, ped = run_gpu(case, cases.make_input(case))
    want = golden[name + "__tps"]
    if case["kind"] == "overflow":
        assert tps.size == want.size == 1
        for f in ("time_start", "time_peak", "time_over_threshold", "adc_peak", "channel"):
            assert tps[0][f] == want[0][f]
        assert (tps[0]["adc_integral"], want[0]["adc_integral"]) == (59990, 32767)
    else:
        assert_same_tps(tps, want, name)
    assert (ped == golden[name + "__pedestal"]).all()


@pytest.mark.parametrize("fmt", ["wibeth", "wib2"])
@pytest.mark.parametrize("thr", [5, 6, 7, 9, 11, 40])
def test_fir_thresholds_beyond_the_packed_comparator_range(fmt, thr):
    """sigma * multiplier * threshold is compared as a SIGNED int16 by the reference (_mm256_cmpgt_epi16 on the 16-bit lanes of a
    64-bit-lane product, wib2/tpg/ProcessAVX2FIR.hpp:208): with multiplier 64 it goes negative once sigma * threshold > 511,
    i.e. for threshold >= 6 on a channel whose IQR reaches 57..86 — is_over is then true for almost every sample and the
    charge takes an arithmetic shift of a possibly negative filter output. Wide noise (sigma at its clamp of 102) puts every
    channel there; 102 * 64 * 5 = 32640 is the last product the packed comparator handles, everything above runs the
    exact-threshold tier. TPs, quartiles and the FIR ring must match the oracle (pinned to the reference for these inputs by
    tests/test_oracle_vs_reference.py::test_fir_threshold_64bit_lane_product and the wib2_fir_thr*_noisy golden cases)."""
    p = S.gen_params(61, 0.3, noise_q8=40 * 256)
    n_links, n_units = 3, 40
    units = (S.gen_wib2_host if fmt == "wib2" else S.gen_wibeth_host)(p, n_links, n_units)
    cfg = B.make_config(fmt=fmt, algorithm=S.ALGORITHMS["FIR"], threshold=thr)
    want, oracles = B.oracle_process_links(cfg, units)
    with S.TPGenerator(n_links, 16, fmt=fmt, algorithm="FIR", threshold=thr, tp_capacity=1 << 20) as g:
        g.start()
        parts = [g.process_host(np.ascontiguousarray(units[:, u:u + 16]), units_stride=min(16, n_units - u)) for u in range(0, n_units, 16)]
        got = np.concatenate(parts)
        assert got.size > 20
        assert_same_tps(got, want, f"{fmt} FIR thr {thr}")
        assert_same_state(g.dump_state(1)[None], oracles[1].state()[None], fmt, "FIR", f"{fmt} FIR thr {thr}, link 1")


def test_unpack_known_answer_through_the_abi():
    """unittest/WIBEthFrameExpansion_test.cxx:92-156 and test/apps/wib2_test_bench.cxx:233-254 on the CUDA path: a frame whose
    ADC value IS its channel number. The pedestal is seeded with the first sample and never moves on a constant input, so the
    per-sample pedestal dump of swtpg_process_host_debug is the unpacked frame, by FRAME channel (the lane permutation of the
    AVX2 registers, H1, does not exist on this path), and the pedestal-subtracted waveform is zero."""
    with S.TPGenerator(1, 1, threshold=60) as g:
        g.start()
        tps, ped, wav = g.process_host(cases.unpack_kat_frame()[None, None], debug=True)
        assert tps.size == 0
        assert (ped[0, 0] == np.arange(64, dtype=np.int16)[None, :]).all() and not wav.any()
        assert (g.dump_state(0)["pedestal"] == np.arange(64)).all()
    with S.TPGenerator(1, 1, fmt="wib2", threshold=60) as g:
        g.start()
        tps, ped, wav = g.process_host(cases.unpack_kat_superchunk()[None, None], debug=True)
        assert tps.size == 0
        assert (ped[0, 0] == (0x3A0 + np.arange(256, dtype=np.int16))[None, :]).all() and not wav.any()
    # every 14-bit value at every bit offset of the row: channel c carries (5 * 64 * t + 321 * c) mod 2^14 at tick t
    adc = ((5 * 64 * np.arange(64)[:, None] + 321 * np.arange(64)[None, :]) % 16384).astype(np.uint16)
    fr = F.pack_wibeth_frames(adc[None], 7)[0]
    with S.TPGenerator(1, 1, threshold=16383) as g:
        g.start()
        _, ped, wav = g.process_host(fr[None, None], debug=True)
        assert ((ped[0, 0].astype(np.int32) + wav[0, 0]) == adc).all()  # pedestal + (sample - pedestal) = the unpacked sample


@pytest.mark.parametrize("name", ["noise_simple_thr60", "dense_simple_thr8", "noise_absrs_thr30", "wib2_simple_thr100", "wib2_fir_thr5", "wib2_absrs_thr60"])
@pytest.mark.parametrize("max_units", [1, 7, 32])
def test_batching_does_not_change_results(name, max_units, golden):
    """Superchunk length is an implementation choice: state carried across batches must make it invisible."""
    case = cases.GOLDEN_CASES[name]
    tps, ped = run_gpu(case, cases.make_input(case), max_units=max_units)
    assert_same_tps(tps, golden[name + "__tps"], f"{name} max_units={max_units}")
    assert (ped == golden[name + "__pedestal"]).all()


@pytest.mark.parametrize("algorithm,thr,L", [("SimpleThreshold", 25, 10), ("SimpleThreshold", 0, 1), ("SimpleThreshold", 25, 0),
                                              ("SimpleThreshold", 40000, 10), ("SimpleThreshold", 25, -3), ("SimpleThreshold", 12, 300),
                                              ("AbsRS", 30, 10), ("StandardRS", 30, 4), ("FIR", 5, 10), ("FIR", 40, 10)])
def test_against_oracle_with_state_and_dumps(algorithm, thr, L):
    """Random waveforms, several links, 3 batches (last one short): TPs, every carried state field, and the per-sample
    pedestal / filtered-waveform dumps equal the oracle's. Covers the packed fast path (L >= 1, thr <= 32767) and the
    scalar path (degenerate accumulator limits, thresholds >= 2^15 that the reference compares as negative int16)."""
    n_links, n_units = 5, 20
    units = S.gen_wibeth_host(S.gen_params(41, 0.4), n_links, n_units)
    cfg = B.make_config(algorithm=S.ALGORITHMS[algorithm], threshold=thr, acc_limit=L)
    oracles = [B.Oracle(cfg, link_id=l) for l in range(n_links)]
    want, peds, wavs = [], [], []
    for l in range(n_links):
        t, p, w = oracles[l].process(units[l], dump=True, cap=1 << 20)
        want.append(t), peds.append(p), wavs.append(w)
    got, gp, gw = [], [], []
    with S.TPGenerator(n_links, 8, algorithm=algorithm, threshold=thr, acc_limit=L, tp_capacity=1 << 21) as g:
        g.start()
        for u in range(0, n_units, 8):
            t, p, w = g.process_host(np.ascontiguousarray(units[:, u:u + 8]), debug=True, cap=1 << 21)
            got.append(t), gp.append(p), gw.append(w)
        assert_same_tps(np.concatenate(got), np.concatenate(want), algorithm)
        assert (np.concatenate(gp, axis=1) == np.stack(peds)).all(), "pedestal dump"
        assert (np.concatenate(gw, axis=1) == np.stack(wavs)).all(), "waveform dump"
        assert_same_state(dump_states(g), np.stack([o.state() for o in oracles]), "wibeth", algorithm, algorithm)


ANY_TAPS = [([2, 5, 11, 17, 9, 4, 1], 6), ([-3, 7, 20, 31, 20, 7, -3], 6), ([1, 3, 8, 10, 8, 3, 1], 5), ([300, -700, 1200, 2000, 1200, -700, 300], 6)]


@pytest.mark.parametrize("fmt", ["wibeth", "wib2"])
@pytest.mark.parametrize("taps,exponent", ANY_TAPS)
def test_fir_with_arbitrary_taps(fmt, taps, exponent):
    """FIR + IQR with taps other than firwin_int(7, 0.1, 64) — another multiplier, an asymmetric filter, negative and large taps
    whose products wrap in 16 bits — runs the packed multiply-add policy (PackedFirIqrAnyTaps), not the scalar fallback:
    TPs, filtered-waveform dump, ring state and quartiles equal the oracle (which tests/test_oracle_vs_reference.py pins
    against the reference's own ProcessingInfo with the same taps). Three ragged batches, so the ring phase is carried."""
    n_links, n_units, step = 3, 40, 16
    if fmt == "wib2":
        units = S.gen_wib2_host(S.gen_params(52, 0.5), n_links, n_units)
    else:
        units = S.gen_wibeth_host(S.gen_params(52, 0.5), n_links, n_units)
    cfg = B.make_config(fmt=fmt, algorithm=S.ALGORITHMS["FIR"], threshold=5, fir_taps=taps, tap_exponent=exponent)
    oracles = [B.Oracle(cfg, link_id=l) for l in range(n_links)]
    want, peds, wavs = [], [], []
    for l in range(n_links):
        t, p, w = oracles[l].process(units[l], dump=True, cap=1 << 21)
        want.append(t), peds.append(p), wavs.append(w)
    got, gp, gw = [], [], []
    with S.TPGenerator(n_links, step, fmt=fmt, algorithm="FIR", threshold=5, fir_taps=taps, tap_exponent=exponent, tp_capacity=1 << 22) as g:
        g.start()
        for u in range(0, n_units, step):
            t, p, w = g.process_host(np.ascontiguousarray(units[:, u:u + step]), debug=True, cap=1 << 22)
            got.append(t), gp.append(p), gw.append(w)
        assert (np.concatenate(gw, axis=1) == np.stack(wavs)).all(), "waveform dump"
        assert (np.concatenate(gp, axis=1) == np.stack(peds)).all(), "pedestal dump"
        assert_same_tps(np.concatenate(got), np.concatenate(want), f"{fmt} taps {taps}")
        assert_same_state(dump_states(g), np.stack([o.state() for o in oracles]), fmt, "FIR", f"{fmt} taps {taps}")


@pytest.mark.parametrize("algorithm,thr", [("SimpleThreshold", 30), ("SimpleThreshold", 2), ("SimpleThreshold", 40000), ("FIR", 5), ("FIR", 2),
                                           ("AbsRS", 60), ("AbsRS", 3), ("AbsRS", 700)])
def test_wib2_against_oracle_with_state_and_dumps(algorithm, thr):
    """BASELINE config 5: WIB2 superchunks (256 channels x 12 ticks) through the same fused kernels — SimpleThreshold with the
    >>6 charge (wib2/tpg/ProcessAVX2.hpp) and the FIR + IQR finder (wib2/tpg/ProcessAVX2FIR.hpp). Ragged batches, several
    links; TPs, carried state and per-sample pedestal / waveform dumps equal the oracle's."""
    n_links, n_units, step = 3, 50, 16
    units = S.gen_wib2_host(S.gen_params(51, 0.5), n_links, n_units)
    cfg = B.make_config(fmt="wib2", algorithm=S.ALGORITHMS[algorithm], threshold=thr)
    oracles = [B.Oracle(cfg, link_id=l) for l in range(n_links)]
    want, peds, wavs = [], [], []
    for l in range(n_links):
        t, p, w = oracles[l].process(units[l], dump=True, cap=1 << 20)
        want.append(t), peds.append(p), wavs.append(w)
    got, gp, gw = [], [], []
    with S.TPGenerator(n_links, step, fmt="wib2", algorithm=algorithm, threshold=thr, tp_capacity=1 << 21) as g:
        g.start()
        for u in range(0, n_units, step):
            t, p, w = g.process_host(np.ascontiguousarray(units[:, u:u + step]), debug=True, cap=1 << 21)
            got.append(t), gp.append(p), gw.append(w)
        assert_same_tps(np.concatenate(got), np.concatenate(want), f"wib2 {algorithm}")
        assert (np.concatenate(gp, axis=1) == np.stack(peds)).all(), "pedestal dump"
        assert (np.concatenate(gw, axis=1) == np.stack(wavs)).all(), "waveform dump"
        assert_same_state(dump_states(g), np.stack([o.state() for o in oracles]), "wib2", algorithm, f"wib2 {algorithm}")


@pytest.mark.parametrize("fmt,algorithm,thr,kw", [
    ("wibeth", "SimpleThreshold", 100, {}), ("wibeth", "AbsRS", 100, dict(rs_memory_factor=8, rs_scale_factor=5)),
    ("wibeth", "AbsRS", 50, dict(rs_memory_factor=9, rs_scale_factor=10)), ("wibeth", "StandardRS", 100, dict(rs_memory_factor=7, rs_scale_factor=2)),
    ("wibeth", "FIR", 5, {}), ("wib2", "SimpleThreshold", 100, {}), ("wib2", "FIR", 5, {}), ("wib2", "AbsRS", 40, {})])
def test_extreme_amplitudes_wrap_and_saturate_like_the_reference(fmt, algorithm, thr, kw):
    """Pulses up to the full 14-bit range on low pedestals, dense, bipolar: charge wraps (SimpleThreshold, H3) or saturates
    (RS / WIB2 / FIR), |s'| * scale and RS * R overflow 16 bits, the FIR sum wraps, the input clamp at adcMax and the
    sigma clamp at sigmaMax engage, hits span many frames. The packed fast paths must wrap / saturate bit for bit like the
    reference arithmetic (oracle); per-channel RS memory factors include 0 and odd values."""
    n_links, n_units, step = 2, 24 if fmt == "wibeth" else 120, 8 if fmt == "wibeth" else 40
    p = S.gen_params(71, 0.9, amp_min=3000, amp_max=15000, hw_min=6, hw_max=16, ped_base=300, ped_step=3, noise_q8=40 * 256)
    units = (S.gen_wib2_host if fmt == "wib2" else S.gen_wibeth_host)(p, n_links, n_units)
    cfg = B.make_config(fmt=fmt, algorithm=S.ALGORITHMS[algorithm], threshold=thr, **kw)
    nch = 256 if fmt == "wib2" else 64
    factors = (np.arange(n_links * nch, dtype=np.uint16) * 7 % 13).reshape(n_links, nch)  # 0..12, incl. 0
    oracles = [B.Oracle(cfg, link_id=l) for l in range(n_links)]
    want, peds, wavs = [], [], []
    for l in range(n_links):
        if "RS" in algorithm and fmt == "wibeth":
            oracles[l].set_memory_factor(factors[l])
        t, pd, w = oracles[l].process(units[l], dump=True, cap=1 << 20)
        want.append(t), peds.append(pd), wavs.append(w)
    got, gp, gw = [], [], []
    with S.TPGenerator(n_links, step, fmt=fmt, algorithm=algorithm, threshold=thr, tp_capacity=1 << 21, **kw) as g:
        if "RS" in algorithm and fmt == "wibeth":
            g.set_rs_memory_factor(factors)
        g.start()
        for u in range(0, n_units, step):
            t, pd, w = g.process_host(np.ascontiguousarray(units[:, u:u + step]), debug=True, cap=1 << 21)
            got.append(t), gp.append(pd), gw.append(w)
        assert (np.concatenate(gp, axis=1) == np.stack(peds)).all(), "pedestal dump"
        assert (np.concatenate(gw, axis=1) == np.stack(wavs)).all(), "waveform dump"
        assert_same_tps(np.concatenate(got), np.concatenate(want), f"{fmt} {algorithm}")
        assert_same_state(dump_states(g), np.stack([o.state() for o in oracles]), fmt, algorithm, f"{fmt} {algorithm}")
    allt = np.concatenate(want)
    assert allt.size > 200
    if algorithm == "SimpleThreshold" and fmt == "wibeth":
        assert (allt["adc_integral"] > 40000).any(), "no wrapped charge in the sample: the case does not test H3"


@pytest.mark.parametrize("algorithm", ["AbsRS", "StandardRS"])
def test_per_link_memory_factor_after_start(algorithm):
    """swtpg_set_link_rs_memory_factor: what a frame processor calls from find_hits on ITS first frame (the per-plane factors of
    src/wibeth/WIBEthFrameProcessor.cpp:437-456 depend on the frame's geo id) — after start, one link at a time, from that link's
    own thread, while other links are already running. One small asynchronous copy per call, ordered on the compute stream;
    only that link's rows change. Links 0 and 2 set theirs before their first unit, link 1 keeps the configured factor, link 3
    sets it after its first batch (the new factor applies from the next batch on, the carried running sum stays)."""
    import threading

    n_links, n_units, step = 4, 24, 8
    units = S.gen_wibeth_host(S.gen_params(73, 0.5), n_links, n_units)
    cfg = B.make_config(algorithm=S.ALGORITHMS[algorithm], threshold=30, rs_memory_factor=8, rs_scale_factor=5)
    fac = {l: ((np.arange(64, dtype=np.uint16) * (3 + l)) % 11).astype(np.uint16) for l in (0, 2, 3)}
    oracles = [B.Oracle(cfg, link_id=l) for l in range(n_links)]
    want = []
    for l in range(n_links):
        if l in (0, 2):
            oracles[l].set_memory_factor(fac[l])
        want.append(oracles[l].process(units[l, :step]))
        if l == 3:
            oracles[l].set_memory_factor(fac[l])
        want.append(oracles[l].process(units[l, step:]))
    with S.TPGenerator(n_links, step, algorithm=algorithm, threshold=30, rs_memory_factor=8, rs_scale_factor=5, tp_capacity=1 << 20) as g:
        g.start()
        th = [threading.Thread(target=g.set_link_rs_memory_factor, args=(l, fac[l])) for l in (0, 2)]  # concurrently, as link threads do
        for t in th:
            t.start()
        for t in th:
            t.join()
        got = [g.process_host(np.ascontiguousarray(units[:, :step]))]
        g.set_link_rs_memory_factor(3, fac[3])
        for u in range(step, n_units, step):
            got.append(g.process_host(np.ascontiguousarray(units[:, u:u + step])))
        assert_same_tps(np.concatenate(got), np.concatenate(want), "per-link memory factor")
        assert_same_state(dump_states(g), np.stack([o.state() for o in oracles]), "wibeth", algorithm, "per-link memory factor")


def test_wib2_many_links_ragged_and_streaming():
    """More links than one wave of CTAs would be on a small grid, ragged unit counts, then the streaming entry points."""
    n_links, stride = 9, 8
    units = S.gen_wib2_host(S.gen_params(52, 0.4), n_links, 2 * stride)
    nu = np.array([8, 0, 3, 8, 1, 8, 5, 8, 2], dtype=np.uint32)
    cfg = B.make_config(fmt="wib2", threshold=25)
    want = []
    for l in range(n_links):
        o = B.Oracle(cfg, link_id=l)
        want += [o.process(units[l, : nu[l]]), o.process(units[l, stride:])]
    with S.TPGenerator(n_links, stride, fmt="wib2", threshold=25) as g:
        g.start()
        a = g.process_host(np.ascontiguousarray(units[:, :stride]), n_units=nu)
        b = g.process_host(np.ascontiguousarray(units[:, stride:]))
        assert_same_tps(np.concatenate([a, b]), np.concatenate(want), "wib2 ragged")
    want2, _ = B.oracle_process_links(cfg, units)
    got = []
    with S.TPGenerator(n_links, 4, fmt="wib2", threshold=25, n_slots=3) as g:
        g.start()
        for u in range(2 * stride):
            for l in range(n_links):
                while not g.submit(l, units[l, u]):
                    got.append(g.poll())
            got.append(g.poll())
        got.append(g.drain())  # flush + sync + poll until the library reports nothing pending, in flight or ready
    assert_same_tps(np.concatenate(got), want2, "wib2 streaming")


def test_wib2_standard_rs_does_not_exist():
    with pytest.raises(S.SwtpgError) as e:
        S.TPGenerator(1, 4, fmt="wib2", algorithm="StandardRS")
    assert e.value.status == 6  # SWTPG_ERR_UNSUPPORTED (reference: TPGAlgorithmInexistent)
    with pytest.raises(S.SwtpgError) as e:
        S.TPGenerator(1, 4, fmt="wib2", algorithm="AbsRS", threshold=0)
    assert e.value.status == 1  # the reference would divide by zero (sigmaMax)


def test_ragged_and_empty_batches():
    """n_units per link: 0, 1, full and in between; an all-empty batch is a no-op."""
    n_links, stride = 6, 10
    units = S.gen_wibeth_host(S.gen_params(43, 0.5), n_links, 2 * stride)
    nu1 = np.array([0, 1, 10, 3, 10, 7], dtype=np.uint32)
    nu2 = np.array([10, 0, 5, 10, 2, 9], dtype=np.uint32)
    cfg = B.make_config(threshold=20)
    want = []
    for l in range(n_links):
        o = B.Oracle(cfg, link_id=l)
        want += [o.process(units[l, : nu1[l]]), o.process(units[l, stride: stride + nu2[l]])]
    with S.TPGenerator(n_links, stride, threshold=20) as g:
        g.start()
        a = g.process_host(np.ascontiguousarray(units[:, :stride]), n_units=nu1)
        e = g.process_host(np.ascontiguousarray(units[:, :stride]), n_units=np.zeros(n_links, dtype=np.uint32))
        z = g.process_host(np.zeros((n_links, 0, 7200), dtype=np.uint8), units_stride=0)
        b = g.process_host(np.ascontiguousarray(units[:, stride:]), n_units=nu2)
        assert e.size == 0 and z.size == 0
        assert_same_tps(np.concatenate([a, b]), np.concatenate(want), "ragged")
        assert g.counters()["units_processed"] == int(nu1.sum() + nu2.sum())


def test_more_links_than_persistent_warps_ragged():
    """Links are handed to the persistent warps through a device-side cursor (wibeth_kernel): more links than the GPU holds
    warps, ragged unit counts with empty links in between, several launches on one handle (the cursor re-arms itself), and
    two algorithms with different warps-per-SM settings. Every link's TPs and pedestals must equal the oracle's, and every
    link must have been processed exactly once per launch (units_processed)."""
    n_links, stride = 3300, 3
    p = S.gen_params(53, 0.5)
    units = S.gen_wibeth_host(p, n_links, 2 * stride)
    rng = np.random.default_rng(7)
    nus = [rng.integers(0, stride + 1, n_links).astype(np.uint32) for _ in range(2)]
    nus[0][:40] = 0
    nus[1][-5:] = 0
    for algorithm, thr in (("SimpleThreshold", 20), ("FIR", 5)):
        cfg = B.make_config(algorithm=S.ALGORITHMS[algorithm], threshold=thr)
        check = list(range(0, n_links, 97)) + [n_links - 1, 2959, 2960, 2961]
        want, ped = [], {}
        for l in check:
            o = B.Oracle(cfg, link_id=l)
            want += [o.process(units[l, : nus[0][l]]), o.process(units[l, stride: stride + nus[1][l]])]
            ped[l] = o.state()["pedestal"]
        with S.TPGenerator(n_links, stride, algorithm=algorithm, threshold=thr, tp_capacity=1 << 22) as g:
            g.start()
            a = g.process_host(np.ascontiguousarray(units[:, :stride]), n_units=nus[0])
            b = g.process_host(np.ascontiguousarray(units[:, stride:]), n_units=nus[1])
            got = np.concatenate([a, b])
            assert g.counters()["units_processed"] == int(nus[0].sum() + nus[1].sum())
            for l in check:
                if nus[0][l] + nus[1][l]:
                    assert (g.dump_state(l)["pedestal"] == ped[l]).all(), f"{algorithm} link {l}"
        assert_same_tps(got[np.isin(got["link"], check)], np.concatenate(want), f"{algorithm} dynamic hand-out")
        # every link with data produced its TPs exactly once: the per-link TP count equals a second, independent run
        with S.TPGenerator(n_links, stride, algorithm=algorithm, threshold=thr, tp_capacity=1 << 22) as g:
            g.start()
            a2 = g.process_host(np.ascontiguousarray(units[:, :stride]), n_units=nus[0])
            b2 = g.process_host(np.ascontiguousarray(units[:, stride:]), n_units=nus[1])
        assert_same_tps(np.concatenate([a2, b2]), got, f"{algorithm} run-to-run")


def test_more_links_than_persistent_warps_whole_batches():
    """The same hand-out with every link carrying the same number of units — the bench's shape: two launches on one handle (the
    cursor and the per-link slice counters re-arm themselves), SimpleThreshold and a running sum, sampled links against the
    oracle incl. their pedestals, and the whole TP list against a second run. Under SWTPG_PARTS (test_links_handed_out_in_slices)
    every link of these batches is handed out in slices."""
    n_links, stride = 4500, 16
    units = S.gen_wibeth_host(S.gen_params(57, 0.05), n_links, 2 * stride)
    for algorithm, thr in (("SimpleThreshold", 20), ("StandardRS", 40)):
        cfg = B.make_config(algorithm=S.ALGORITHMS[algorithm], threshold=thr)
        check = list(range(0, n_links, 211)) + [n_links - 1, 4143, 4144, 4145]
        want, ped = [], {}
        for l in check:
            o = B.Oracle(cfg, link_id=l)
            want.append(o.process(units[l]))
            ped[l] = o.state()["pedestal"]
        runs = []
        for _ in range(2):
            with S.TPGenerator(n_links, stride, algorithm=algorithm, threshold=thr, tp_capacity=1 << 22) as g:
                g.start()
                a = g.process_host(np.ascontiguousarray(units[:, :stride]))
                b = g.process_host(np.ascontiguousarray(units[:, stride:]))
                runs.append(np.concatenate([a, b]))
                assert g.counters()["units_processed"] == 2 * n_links * stride
                for l in check:
                    assert (g.dump_state(l)["pedestal"] == ped[l]).all(), f"{algorithm} link {l}"
        assert_same_tps(runs[0][np.isin(runs[0]["link"], check)], np.concatenate(want), f"{algorithm} whole batches")
        assert_same_tps(runs[1], runs[0], f"{algorithm} run-to-run")


@pytest.mark.skipif(os.environ.get("SWTPG_PARTS") is not None, reason="already running with forced slicing")
@pytest.mark.parametrize("parts", [2, 4, 8])
def test_links_handed_out_in_slices(parts):
    """A launch with more links than persistent warps hands every link out in slices (wibeth_kernel: a later slice continues from
    the state its predecessor stored, and may run on another warp). SWTPG_PARTS forces that for EVERY launch of a process, so
    the ragged / empty / carried-state / dump / hand-out cases above are repeated under it: units fewer than slices (empty
    slices), hits open across a slice boundary, FIR ring phase, running sums, the scalar policies. 4 is the slice count of
    the production launches (tests/test_gpu_launch_geometry.py runs those in their default geometries)."""
    env = dict(os.environ, SWTPG_PARTS=str(parts))
    sel = ("test_more_links_than_persistent_warps_ragged or test_more_links_than_persistent_warps_whole_batches or "
           "test_ragged_and_empty_batches or test_against_oracle_with_state_and_dumps or "
           "test_batching_does_not_change_results or test_extreme_amplitudes_wrap_and_saturate_like_the_reference")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-q", "-x", "-m", "gpu", "-k", sel, "-p", "no:cacheprovider"],
                       env=env, capture_output=True, text=True, cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert " passed" in r.stdout and "failed" not in r.stdout, r.stdout[-2000:]


def test_restart_resets_state():
    """start() = fresh ChanState + first_hit re-armed (src/wibeth/WIBEthFrameProcessor.cpp:111-154, 67-72)."""
    units = S.gen_wibeth_host(S.gen_params(44, 0.5), 2, 12)
    with S.TPGenerator(2, 12, threshold=20) as g:
        g.start()
        a = g.process_host(units)
        g.stop()
        g.start()
        b = g.process_host(units)
        assert_same_tps(a, b, "restart")
        with pytest.raises(S.SwtpgError):
            g.stop()
            g.process_host(units)  # not started


def test_streaming_submit_poll_equals_batch():
    """The drop-in path: per-link submit of single frames, auto-dispatch of full superchunks on the staging ring,
    poll; then flush of the ragged tail. Equals the batch entry point and the oracle."""
    n_links, n_units, sc = 7, 23, 4
    units = S.gen_wibeth_host(S.gen_params(45, 0.5), n_links, n_units)
    want, _ = B.oracle_process_links(B.make_config(threshold=20), units)
    got = []
    with S.TPGenerator(n_links, sc, threshold=20, n_slots=3) as g:
        g.start()
        busy = 0
        for u in range(n_units):
            for l in range(n_links):
                while not g.submit(l, units[l, u]):
                    busy += 1
                    got.append(g.poll())  # back-pressure: drain completed batches, then retry
            got.append(g.poll())
        got.append(g.drain())  # flush + sync + poll until the library reports nothing pending, in flight or ready
        c = g.counters()
        assert c["units_processed"] == n_links * n_units
        assert c["h2d_bytes"] == n_links * n_units * 7200
    assert_same_tps(np.concatenate(got), want, "streaming")


def test_streaming_zero_copy_from_a_registered_latency_buffer():
    """swtpg_register_buffer: payloads submitted from inside a registered array are not copied by submit; the copy engine reads
    them where they lie when the superchunk is dispatched. Link 0 and 1 come straight out of the registered buffer (one
    contiguous run per superchunk), link 2 out of a ring that wraps inside a superchunk (two runs), link 3 from unregistered
    memory (staged copy as before), link 4 alternates between registered and unregistered payloads. Same TPs as the oracle."""
    n_links, n_units, sc = 5, 24, 8
    units = S.gen_wibeth_host(S.gen_params(47, 0.5), n_links, n_units)
    want, _ = B.oracle_process_links(B.make_config(threshold=20), units)
    latency_buffer = units.copy()                       # the registered memory
    ring = np.roll(latency_buffer[2], 3, axis=0).copy() # unit u of link 2 lives at ring[(u + 3) % n_units]
    outside = units.copy()                              # never registered
    got = []
    with S.TPGenerator(n_links, sc, threshold=20, n_slots=3) as g:
        g.register_buffer(latency_buffer)
        g.register_buffer(ring)
        g.start()
        for u in range(n_units):
            srcs = [latency_buffer[0, u], latency_buffer[1, u], ring[(u + 3) % n_units], outside[3, u],
                    latency_buffer[4, u] if u % 3 else outside[4, u]]
            for l, src in enumerate(srcs):
                while not g.submit(l, src):
                    got.append(g.poll())
            got.append(g.poll())
        got.append(g.drain())  # flush + sync + poll until the library reports nothing pending, in flight or ready
        c = g.counters()
        assert c["units_processed"] == n_links * n_units and c["h2d_bytes"] == n_links * n_units * 7200
        # links 0, 1, 2 entirely by address, link 3 entirely by copy, link 4 by address except every third payload
        by_address = 3 * n_units + sum(1 for u in range(n_units) if u % 3)
        assert (c["units_zero_copy"], c["units_staged"]) == (by_address, n_links * n_units - by_address)
        g.unregister_buffer(ring)
        g.unregister_buffer(latency_buffer)
        with pytest.raises(S.SwtpgError):
            g.unregister_buffer(outside)
    assert_same_tps(np.concatenate(got), want, "zero-copy streaming")


def test_streaming_links_out_of_step():
    """Links are fed by independent threads and advance independently: a link that runs superchunks ahead of the others gets its
    TPs while the others are still silent (batches are ragged; there is no all-links barrier), and nothing is lost or
    reordered per link when the stragglers arrive."""
    n_links, n_units, sc = 3, 8, 4
    units = S.gen_wibeth_host(S.gen_params(46, 0.5), n_links, n_units)
    cfg = B.make_config(threshold=20)
    want, _ = B.oracle_process_links(cfg, units)
    want0 = B.Oracle(cfg, link_id=0).process(units[0])
    with S.TPGenerator(n_links, sc, threshold=20, n_slots=2) as g:
        g.start()
        for u in range(n_units):  # link 0 first, all of it; links 1 and 2 deliver nothing yet
            assert g.submit(0, units[0, u], wait_us=2_000_000)
        first = g.drain()
        assert_same_tps(first, want0, "link 0 alone")
        for l in (1, 2):
            for u in range(n_units):
                assert g.submit(l, units[l, u], wait_us=2_000_000)
        rest = g.drain()
        assert g.counters()["units_processed"] == n_links * n_units
    assert_same_tps(np.concatenate([first, rest]), want, "out of step")


def test_streaming_back_pressure_is_busy_not_blocking():
    """Nobody polls: after n_slots batches hold un-polled TPs the dispatcher stalls, the link's ring (n_slots superchunks)
    fills up and swtpg_submit answers BUSY instead of blocking; flush reports the same condition. Polling releases everything."""
    n_slots, sc = 2, 4
    units = S.gen_wibeth_host(S.gen_params(48, 0.5), 1, 6 * sc)
    want = B.Oracle(B.make_config(threshold=20)).process(units[0])
    got = []
    with S.TPGenerator(1, sc, threshold=20, n_slots=n_slots) as g:
        g.start()
        accepted = 0
        for u in range(units.shape[1]):
            for _ in range(200):  # up to 200 ms per unit for batches to be dispatched and rings to be released
                if g.submit(0, units[0, u]):
                    accepted += 1
                    break
                time.sleep(0.001)
            else:
                break
        assert n_slots * sc <= accepted <= 2 * n_slots * sc, accepted  # n_slots batches + at most one ring of pending units
        assert accepted < units.shape[1]
        assert g.counters()["submit_busy"] > 0
        assert not g.flush(busy_ok=True)  # every batch waits to be polled
        got.append(g.drain())
        for u in range(accepted, units.shape[1]):
            assert g.submit(0, units[0, u], wait_us=2_000_000)
        got.append(g.drain())
    assert_same_tps(np.concatenate(got), want, "after back-pressure")


def test_streaming_partial_superchunks_go_out_after_the_timeout():
    """No link ever fills a superchunk and nobody flushes: pending units are dispatched after dispatch_timeout_us."""
    n_links, n_units = 4, 5
    units = S.gen_wibeth_host(S.gen_params(49, 0.5), n_links, n_units)
    want, _ = B.oracle_process_links(B.make_config(threshold=20), units)
    got = []
    with S.TPGenerator(n_links, 64, threshold=20, dispatch_timeout_us=20_000) as g:
        g.start()
        for u in range(n_units):
            for l in range(n_links):
                assert g.submit(l, units[l, u])
        deadline = time.time() + 5.0
        while g.counters()["units_processed"] < n_links * n_units and time.time() < deadline:
            got.append(g.poll(wait_us=50_000))
        assert g.counters()["units_processed"] == n_links * n_units
        g.sync()
        for _ in range(4):
            got.append(g.poll())
    assert_same_tps(np.concatenate(got), want, "time-out dispatch")


def test_streaming_concurrent_feeders_and_flushes():
    """Feeder threads submit while another thread keeps flushing (a watchdog): flush is safe against concurrent submits."""
    import threading

    n_links, n_units, sc = 12, 96, 8
    units = S.gen_wibeth_host(S.gen_params(50, 0.3), n_links, n_units)
    want, _ = B.oracle_process_links(B.make_config(threshold=25), units)
    got, stop = [], threading.Event()
    with S.TPGenerator(n_links, sc, threshold=25, n_slots=3) as g:
        g.start()

        def feed(t):
            for u in range(n_units):
                for l in range(t, n_links, 3):
                    assert g.submit(l, units[l, u], wait_us=5_000_000)

        def watchdog():
            while not stop.is_set():
                g.flush(busy_ok=True)
                time.sleep(0.0005)

        def poller():
            while not stop.is_set():
                got.append(g.poll(wait_us=2000))

        th = [threading.Thread(target=feed, args=(t,)) for t in range(3)] + [threading.Thread(target=watchdog), threading.Thread(target=poller)]
        for t in th:
            t.start()
        for t in th[:3]:
            t.join()
        stop.set()
        for t in th[3:]:
            t.join()
        got.append(g.drain())
        assert g.counters()["units_processed"] == n_links * n_units
    assert_same_tps(np.concatenate(got), want, "concurrent feeders + flushes")


def test_tp_buffer_overflow_is_reported():
    units = S.gen_wibeth_host(S.gen_params(47, 0.9), 2, 8)
    with S.TPGenerator(2, 8, threshold=5, tp_capacity=16) as g:
        g.start()
        with pytest.raises(S.SwtpgError) as e:
            g.process_host(units)
        assert e.value.status == 4  # SWTPG_ERR_OVERFLOW
        c = g.counters()
        assert c["tps_emitted"] > 16 and c["tps_dropped_overflow"] == c["tps_emitted"] - 16


def test_device_generator_matches_host_generator():
    import torch

    p = S.gen_params(48, 0.3)
    n_links, n_units = 9, 5
    buf = torch.empty(n_links * n_units * 7200, dtype=torch.uint8, device="cuda")
    S.gen_wibeth_device(p, buf.data_ptr(), n_links, n_units, link0=4, unit0=3)
    torch.cuda.synchronize()
    host = S.gen_wibeth_host(p, n_links, n_units, link0=4, unit0=3)
    assert (buf.cpu().numpy().reshape(host.shape) == host).all()
    buf2 = torch.empty(3 * 4 * 5664, dtype=torch.uint8, device="cuda")
    S.gen_wib2_device(p, buf2.data_ptr(), 3, 4, link0=2)
    torch.cuda.synchronize()
    host2 = S.gen_wib2_host(p, 3, 4, link0=2)
    assert (buf2.cpu().numpy().reshape(host2.shape) == host2).all()


def test_sharded_equals_unsharded():
    """Links split over two handles (as over two GPUs) + host merge == one handle over all links."""
    from fdreadoutlibs_b200 import sharding

    n_links, n_units = 80, 6
    p = S.gen_params(49, 0.3)
    with S.TPGenerator(n_links, n_units, threshold=30) as g:
        g.start()
        full = S.sort_tps(g.process_host(S.gen_wibeth_host(p, n_links, n_units)))
    parts = []
    for rank in range(2):
        l0, n = sharding.shard_links(n_links, 2, rank)
        with S.TPGenerator(n, n_units, threshold=30) as g:
            g.start()
            parts.append(S.sort_tps(sharding.globalise(g.process_host(S.gen_wibeth_host(p, n, n_units, link0=l0)), l0)))
    merged = S.merge_sorted(parts)
    assert merged.size == full.size and (merged == full).all()


def test_full_size_one_apa_properties():
    """BASELINE config 2 at full size — 40 links x 8192 frames (2.36 GB, 1.34 G samples), resident in HBM.
    Size-independent properties: (1) one 8192-frame batch and 16 batches of 512 give the identical TP multiset;
    (2) two complete links agree with the CPU oracle tuple for tuple; (3) a second start() reproduces the same list."""
    import torch

    n_links, n_units = 40, 8192
    p = S.gen_params(2, 0.02)
    buf = torch.empty(n_links * n_units * 7200, dtype=torch.uint8, device="cuda")
    S.gen_wibeth_device(p, buf.data_ptr(), n_links, n_units)
    torch.cuda.synchronize()
    with S.TPGenerator(n_links, n_units, threshold=60, tp_capacity=1 << 22) as g:
        g.start()
        g.process_device(buf.data_ptr(), n_units)
        one = g.fetch_tps(cap=1 << 22)
        g.stop()
        g.start()
        g.process_device(buf.data_ptr(), n_units)
        again = g.fetch_tps(cap=1 << 22)
    assert one.size > 10000
    assert_same_tps(one, again, "restart determinism")
    # batched: link-major layout with stride 8192 -> batches address sub-ranges by offsetting the base pointer
    parts = []
    with S.TPGenerator(n_links, n_units, threshold=60, tp_capacity=1 << 22) as g:
        g.start()
        view = buf.view(n_links, n_units, 7200)
        ts = torch.cuda.current_stream().cuda_stream  # run on torch's stream: ordered after the .contiguous() copy
        for b in range(16):
            chunk = view[:, b * 512:(b + 1) * 512].contiguous()
            g.process_device(chunk.data_ptr(), 512, stream=ts)
            parts.append(g.fetch_tps(cap=1 << 22))
    assert_same_tps(np.concatenate(parts), one, "batch split")
    cfg = B.make_config(threshold=60)
    for l in (0, 39):
        host = buf.view(n_links, n_units, 7200)[l].cpu().numpy()
        want = B.Oracle(cfg, link_id=l).process(host, cap=1 << 20)
        assert_same_tps(one[one["link"] == l], want, f"link {l} vs oracle")
    # BASELINE config[1] names the FIR kernel: the same properties for the fused unpack -> pedestal -> FIR -> hit-find kernel
    with S.TPGenerator(n_links, n_units, algorithm="FIR", threshold=5, tp_capacity=1 << 22) as g:
        g.start()
        g.process_device(buf.data_ptr(), n_units)
        fir_one = g.fetch_tps(cap=1 << 22)
    parts = []
    with S.TPGenerator(n_links, n_units, algorithm="FIR", threshold=5, tp_capacity=1 << 22) as g:
        g.start()
        view = buf.view(n_links, n_units, 7200)
        ts = torch.cuda.current_stream().cuda_stream
        for b in range(16):
            chunk = view[:, b * 512:(b + 1) * 512].contiguous()
            g.process_device(chunk.data_ptr(), 512, stream=ts)
            parts.append(g.fetch_tps(cap=1 << 22))
    assert fir_one.size > 10000
    assert_same_tps(np.concatenate(parts), fir_one, "FIR batch split")
    fcfg = B.make_config(algorithm=S.ALGORITHMS["FIR"], threshold=5)
    for l in (3, 38):
        host = buf.view(n_links, n_units, 7200)[l].cpu().numpy()
        want = B.Oracle(fcfg, link_id=l).process(host, cap=1 << 20)
        assert_same_tps(fir_one[fir_one["link"] == l], want, f"FIR link {l} vs oracle")


@pytest.mark.parametrize("thr", cases.CONFIG1_THRESHOLDS)
def test_config1_single_link_10k_frames(thr):
    """BASELINE config[0]: one WIBEth link (64 ch x 64 ticks/frame), 10 000 synthetic frames (40.96 M samples), SimpleThreshold,
    accumulator limit 10 — the run the reference's (absent) emulator app would do with AVX and NAIVE implementations.
    GPU == AVX2 flavour on every field; == what the reference's own compiled code returned (tests/golden/reference_outputs.npz);
    == NAIVE flavour after its position->channel mapping wherever the integral did not overflow 15 bits (SURVEY H1, H3)."""
    n_frames = 10000
    units = cases.config1_input()
    assert units.shape[1] == n_frames
    with S.TPGenerator(1, 2500, threshold=thr, tp_capacity=1 << 20) as g:
        g.start()
        got = np.concatenate([g.process_host(np.ascontiguousarray(units[:, u:u + 2500])) for u in range(0, n_frames, 2500)])
        ped = g.dump_state(0)["pedestal"]
    o = B.Oracle(B.make_config(threshold=thr))
    want = o.process(units[0], cap=1 << 20)
    assert want.size > 3000
    assert_same_tps(got, want, "AVX2 flavour")
    assert (ped == o.state()["pedestal"]).all()
    naive = B.Oracle(B.make_config(threshold=thr), B.FLAVOUR_NAIVE).process(units[0], cap=1 << 20)
    keep = lambda a: a[a["adc_integral"] <= 32767]
    assert_same_tps(keep(got), keep(naive), "NAIVE flavour (integrals <= 32767)")
    assert_same_as_reference({"tps": got}, cases.reference_outputs(), f"config1_thr{thr}")  # process_window_avx2 itself


@pytest.mark.parametrize("algorithm,impl", [("AbsRS", B.REF_ETH_ABSRS_AVX2), ("StandardRS", B.REF_ETH_STDRS_AVX2)])
def test_running_sums_against_the_reference_itself(algorithm, impl):
    """GPU vs what the reference's own process_window_rs_avx2 / process_window_standard_rs_avx2 (compiled from its headers)
    returned for this input (tests/golden/reference_outputs.npz), no restatement in between."""
    assert algorithm in cases.GPU_RS_DIFF
    units = cases.gpu_rs_input()
    with S.TPGenerator(1, 100, algorithm=algorithm, threshold=30, rs_memory_factor=8, rs_scale_factor=5) as g:
        g.start()
        got = np.concatenate([g.process_host(np.ascontiguousarray(units[:, u:u + 100])) for u in range(0, 300, 100)])
    assert got.size > 500
    assert_same_as_reference({"tps": got}, cases.reference_outputs(), f"gpu_rs_{algorithm}")


@pytest.mark.parametrize("algorithm,impl,thr", [("SimpleThreshold", B.REF_WIB2_SIMPLE_AVX2, 60), ("FIR", B.REF_WIB2_FIR_AVX2, 5)])
def test_wib2_against_the_reference_itself(algorithm, impl, thr):
    """BASELINE config[4]: GPU vs what the reference's own swtpg_wib2::process_window_avx2 (SimpleThreshold and FIR + IQR), both
    register selectors, returned for this input (tests/golden/reference_outputs.npz)."""
    assert (algorithm, thr) in cases.GPU_WIB2_DIFF
    units = cases.gpu_wib2_input()
    with S.TPGenerator(1, 200, fmt="wib2", algorithm=algorithm, threshold=thr) as g:
        g.start()
        got = np.concatenate([g.process_host(np.ascontiguousarray(units[:, u:u + 200])) for u in range(0, 600, 200)])
    assert got.size > 300
    assert_same_as_reference({"tps": got}, cases.reference_outputs(), f"gpu_wib2_{algorithm}_thr{thr}")

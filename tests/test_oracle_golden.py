"""CPU: pins oracle/swtpg_oracle.c against the reference-generated golden vectors (tests/golden/reference_vectors.npz),
the reference's unpack unit test and the TP values its documentation publishes. No GPU, no /root/reference needed."""
import numpy as np
import pytest

import cases
import fdreadoutlibs_b200 as S
from fdreadoutlibs_b200 import _lib
from fdreadoutlibs_b200 import api as A
from fdreadoutlibs_b200 import frames as F
from oracle import binding as B
from util import assert_same_tps, create_status, oracle_config, state_fields


@pytest.mark.parametrize("name", sorted(cases.GOLDEN_CASES))
def test_oracle_matches_reference_vectors(name, golden):
    case = cases.GOLDEN_CASES[name]
    units = cases.make_input(case)
    cfg = oracle_config(case, B)
    tps, oracles = B.oracle_process_links(cfg, units, flavour=case["flavour"])
    assert_same_tps(tps, golden[name + "__tps"], name)
    ped = np.stack([o.state()["pedestal"] for o in oracles])
    assert (ped == golden[name + "__pedestal"]).all(), f"{name}: final pedestals differ from the reference"


def test_documented_golden_tps():
    """docs/README.md:136-146 prints channel,time_start,ToT,time_peak,adc_integral,adc_peak for the golden pattern.
    This snapshot's code gives ToT 288/256 where the doc prints 256/224 (the doc counts ToT "from 0", :142); every other
    field matches the doc (SURVEY.md §4)."""
    cfg = B.make_config(threshold=499)
    tps = F.sort_tps(B.Oracle(cfg).process(cases.golden_frames()))
    assert tps.size == 2
    assert (tps["channel"] == 0).all()
    assert list(tps["time_start"]) == [79554162068719975, 79554162068722023]
    assert list(tps["time_peak"]) == [79554162068720103, 79554162068722151]
    assert list(tps["adc_integral"]) == [4528, 4021]
    assert list(tps["adc_peak"]) == [506, 505]
    assert list(tps["time_over_threshold"]) == [288, 256]


def test_edge_square_spans_frame_boundary():
    """4 + 5 ticks of 600 ADC across a frame boundary -> one TP, emitted in frame 1 at t_end = 5 with tover 9."""
    cfg = B.make_config(threshold=100)
    tps = B.Oracle(cfg).process(cases.edge_square_frames())
    assert tps.size == 1
    tp = tps[0]
    ts1 = (1 << 32) + 2048
    assert tp["channel"] == 9 and tp["time_over_threshold"] == 9 * 32
    assert tp["time_start"] == ts1 + 32 * (5 - 9)  # starts 4 ticks BEFORE the frame that reports it
    assert tp["adc_integral"] == 9 * 600 and tp["adc_peak"] == 600


def test_documented_pulse_and_edge_patterns():
    """docs/README.md:111-116, hand-derived answers (zero frames: pedestal 0, eight ticks over it never move the frugal median).
    pulse: one tick of 650 on channel 33 at tick 17 of frame 1 -> ends at tick 18 with ToT 1.
    edge left / right: the 8-tick triangle 501 520 540 560 540 520 505 501 across the frame boundary -> ONE TP, reported by the
    second frame, time_start before that frame's timestamp; the peak time counts from the hit start."""
    cfg = B.make_config(threshold=499)
    for flav in (B.FLAVOUR_AVX2, B.FLAVOUR_NAIVE):
        tp = B.Oracle(cfg, flav).process(cases.pulse_frames())
        assert tp.size == 1
        ts1 = (1 << 34) + 2048
        assert (tp[0]["channel"], tp[0]["time_start"], tp[0]["time_over_threshold"], tp[0]["adc_integral"], tp[0]["adc_peak"]) == \
            (33, ts1 + 32 * 17, 32, 650, 650)
        assert tp[0]["time_peak"] == tp[0]["time_start"]
        for frames, ch, ts0, n_first in ((cases.edge_left_frames(), 20, 1 << 35, 5), (cases.edge_right_frames(), 47, 1 << 36, 2)):
            tp = B.Oracle(cfg, flav).process(frames)
            assert tp.size == 1
            t_end = 8 - n_first                              # first tick of frame 1 that is not over threshold any more
            start = ts0 + 2048 + 32 * (t_end - 8)            # = 32 * n_first ticks before frame 1
            assert (tp[0]["channel"], tp[0]["time_start"], tp[0]["time_over_threshold"]) == (ch, start, 8 * 32)
            assert tp[0]["adc_integral"] == sum(cases.EDGE_TRIANGLE) and tp[0]["adc_peak"] == 560
            assert tp[0]["time_peak"] == start + 32 * 3      # 560 is the 4th sample of the pulse


def test_charge_overflow_avx2_wraps_naive_saturates():
    """SURVEY H3: 20 ticks x 3000 ADC -> AVX2 add_epi16 wraps mod 2^16, the scalar code saturates at 32767."""
    frames = cases.overflow_frames()
    avx = B.Oracle(B.make_config(threshold=100), B.FLAVOUR_AVX2).process(frames)
    nai = B.Oracle(B.make_config(threshold=100), B.FLAVOUR_NAIVE).process(frames)
    assert avx.size == 1 and nai.size == 1
    # the frugal pedestal steps up once (11th tick over it): 10 x 3000 + 10 x 2999 = 59990 > 32767, kept mod 2^16
    assert avx[0]["adc_integral"] == 59990
    assert nai[0]["adc_integral"] == 32767
    for f in ("time_start", "time_over_threshold", "adc_peak", "channel"):
        assert avx[0][f] == nai[0][f]


def test_unpack_known_answers(golden):
    """unittest/WIBEthFrameExpansion_test.cxx:92-156 and test/apps/wib2_test_bench.cxx:233-254: lane j of register
    j/16 holds channel 16*(j/16) + {0..7,15,8..14}[j%16]."""
    lib = B.oracle_lib()
    out = np.zeros(4096, dtype=np.uint16)
    fr = cases.unpack_kat_frame()
    lib.oracle_wibeth_expand(fr.ctypes.data, out.ctypes.data)
    regs = out.reshape(4, 64, 16)
    expect = np.array([[16 * r + F.LANE_PERM[l] for l in range(16)] for r in range(4)])
    assert (regs == expect[:, None, :]).all()
    assert (out == golden["unpack_kat_wibeth"]).all()
    sc = cases.unpack_kat_superchunk()
    for sel in (0, 1):
        o2 = np.zeros(8 * 12 * 16, dtype=np.uint16)
        lib.oracle_wib2_expand(sc.ctypes.data, sel, 20, o2.ctypes.data)
        assert (o2 == golden[f"unpack_kat_wib2_sel{sel}"]).all()
        regs2 = o2.reshape(8, 12, 16)
        exp2 = np.array([[0x3A0 + 128 * sel + 16 * b + F.LANE_PERM[l] for l in range(16)] for b in range(8)])
        assert (regs2 == exp2[:, None, :]).all()


def test_fir_taps(golden):
    """firwin_int(7, 0.1, 64) = {1,6,15,20,15,6,1} (src/wib2/WIB2FrameProcessor.cpp:93-94)."""
    taps = np.zeros(7, dtype=np.int16)
    assert B.oracle_lib().oracle_firwin_int(7, 0.1, 64, taps.ctypes.data) == 7
    assert list(taps) == [1, 6, 15, 20, 15, 6, 1]
    assert (taps == golden["firwin_int_7_0p1_64"]).all()


def test_numpy_unpack_agrees_with_oracle():
    import fdreadoutlibs_b200 as S

    fr = S.gen_wibeth_host(S.gen_params(9, 0.1), 1, 2)[0]
    adc, ts = F.unpack_wibeth_frames(fr)
    lib = B.oracle_lib()
    for f in range(2):
        for t in (0, 17, 63):
            row = np.ascontiguousarray(fr[f, 32 + 112 * t: 32 + 112 * (t + 1)])
            got = [lib.oracle_unpack14(row.ctypes.data, c) for c in range(64)]
            assert got == list(adc[f, t])
    assert list(ts) == [1 << 40, (1 << 40) + 2048]


def test_oracle_empty_and_state_carry():
    """Zero units is a no-op; processing in two calls equals one call (state carried like ProcessingInfo)."""
    import fdreadoutlibs_b200 as S

    fr = S.gen_wibeth_host(S.gen_params(3, 0.2), 1, 30)[0]
    cfg = B.make_config(threshold=25)
    one = B.Oracle(cfg).process(fr)
    o = B.Oracle(cfg)
    assert o.process(fr[:0]).size == 0
    two = np.concatenate([o.process(fr[:13]), o.process(fr[13:])])
    assert_same_tps(two, one, "split")


# every (format, algorithm) swtpg_create accepts (WIB2 has no StandardRS)
ACCEPTED = [(fmt, a) for fmt in A.FORMATS for a in S.ALGORITHMS if create_status(fmt, a, 30) != _lib.SWTPG_ERR_UNSUPPORTED]


@pytest.mark.parametrize("fmt,algorithm", ACCEPTED)
def test_state_fields_cover_what_moves(fmt, algorithm):
    """util.state_fields, which the GPU tests compare, names every field of the carried state that the oracle moves: every field
    that differs on some channel between the state after the first of 16 generated units and the state after the last. The
    fields left out keep their seeds, such as SimpleThreshold's quartiles and the RS memory factor."""
    gen = S.gen_wib2_host if fmt == "wib2" else S.gen_wibeth_host
    units = gen(S.gen_params(1, 0.3), 1, 16)[0]
    o = B.Oracle(B.make_config(fmt=fmt, algorithm=S.ALGORITHMS[algorithm], threshold=5 if algorithm == "FIR" else 30))
    o.process(units[:1])
    first = o.state()
    o.process(units[1:])
    last = o.state()
    moved = {f for f in F.STATE_DTYPE.names if (first[f] != last[f]).any()}
    assert "pedestal" in moved
    assert moved <= set(state_fields(fmt, algorithm)), f"moved but not compared: {sorted(moved - set(state_fields(fmt, algorithm)))}"

"""Shared test inputs: deterministic frames for the golden cases and the hand-built known-answer patterns.

Patterns follow the reference's documentation of its (absent) pattern generator (docs/README.md:69-146): all five it lists —
"golden" (`500 502 504 505 506 505 504 502 500` on a zero frame, threshold 499), "pulse" (one channel, one tick), "edge square"
(a square pulse across a frame boundary), "edge left" / "edge right" (a triangular pulse spanning two frames with its peak in
the first / second frame) — plus the charge-overflow case of SURVEY.md H3. The doc gives ADC values for "golden" only; the
other shapes are restated from its one-line descriptions.
"""
from __future__ import annotations

import numpy as np

import fdreadoutlibs_b200 as S
from fdreadoutlibs_b200 import frames as F
from oracle import binding as B

GOLDEN_TS0 = 79554162068719943  # docs/README.md:136-146
GOLDEN_PATTERN = [500, 502, 504, 505, 506, 505, 504, 502, 500]


def golden_frames() -> np.ndarray:
    """3 frames, channel 0, pattern at offset 1 of frames 0 and 1 (docs/README.md:86-88)."""
    adc = np.zeros((3, 64, 64), dtype=np.uint16)
    adc[0, 1:10, 0] = GOLDEN_PATTERN
    adc[1, 1:10, 0] = GOLDEN_PATTERN
    return F.pack_wibeth_frames(adc, GOLDEN_TS0)


def edge_square_frames() -> np.ndarray:
    """Square pulse of 600 ADC on channel 9 covering the last 4 ticks of frame 0 and the first 5 of frame 1."""
    adc = np.zeros((3, 64, 64), dtype=np.uint16)
    adc[0, 60:64, 9] = 600
    adc[1, 0:5, 9] = 600
    return F.pack_wibeth_frames(adc, 1 << 32)


def pulse_frames() -> np.ndarray:
    """Single pulse on a single channel and a single tick (docs/README.md:113): 650 ADC on channel 33, tick 17 of frame 1."""
    adc = np.zeros((3, 64, 64), dtype=np.uint16)
    adc[1, 17, 33] = 650
    return F.pack_wibeth_frames(adc, 1 << 34)


EDGE_TRIANGLE = [501, 520, 540, 560, 540, 520, 505, 501]


def edge_left_frames() -> np.ndarray:
    """Triangular pulse spanning two frames, peak in the FIRST frame (docs/README.md:115): channel 20, ticks 59..63 | 0..2."""
    adc = np.zeros((3, 64, 64), dtype=np.uint16)
    adc[0, 59:64, 20] = EDGE_TRIANGLE[:5]  # peak 560 at tick 62
    adc[1, 0:3, 20] = EDGE_TRIANGLE[5:]
    return F.pack_wibeth_frames(adc, 1 << 35)


def edge_right_frames() -> np.ndarray:
    """The same pulse with its peak in the SECOND frame (docs/README.md:116): channel 47, ticks 62..63 | 0..5."""
    adc = np.zeros((3, 64, 64), dtype=np.uint16)
    adc[0, 62:64, 47] = EDGE_TRIANGLE[:2]
    adc[1, 0:6, 47] = EDGE_TRIANGLE[2:]    # peak 560 at tick 1 of frame 1
    return F.pack_wibeth_frames(adc, 1 << 36)


def overflow_frames() -> np.ndarray:
    """Amplitude 3000 for 20 ticks on channel 5 over a flat 100 pedestal: AVX2 charge wraps mod 2^16, naive saturates (H3)."""
    adc = np.full((2, 64, 64), 100, dtype=np.uint16)
    adc[0, 10:30, 5] = 3100
    return F.pack_wibeth_frames(adc, 1 << 33)


def unpack_kat_frame() -> np.ndarray:
    """adc(ch, t) = ch for every tick (unittest/WIBEthFrameExpansion_test.cxx:105-110)."""
    adc = np.tile(np.arange(64, dtype=np.uint16), (1, 64, 1))
    return F.pack_wibeth_frames(adc, 1000)[0]


def unpack_kat_superchunk() -> np.ndarray:
    """adc(ch) = 0x3a0 + ch on every frame of the superchunk (test/apps/wib2_test_bench.cxx:233-236)."""
    adc = np.tile(0x3A0 + np.arange(256, dtype=np.uint16), (12, 1))
    return F.pack_wib2_superchunks(adc, 5000)[0]


# name -> description of a reference-run golden case (tests/golden/make_golden.py). ref_impl codes: oracle/binding.py.
GOLDEN_CASES = {
    "golden_avx2": dict(fmt="wibeth", kind="golden", algorithm="SimpleThreshold", threshold=499, ref_impl=0, flavour=0),
    "golden_naive": dict(fmt="wibeth", kind="golden", algorithm="SimpleThreshold", threshold=499, ref_impl=1, flavour=1),
    "edge_square_avx2": dict(fmt="wibeth", kind="edge", algorithm="SimpleThreshold", threshold=100, ref_impl=0, flavour=0),
    "pulse_avx2": dict(fmt="wibeth", kind="pulse", algorithm="SimpleThreshold", threshold=499, ref_impl=0, flavour=0),
    "pulse_naive": dict(fmt="wibeth", kind="pulse", algorithm="SimpleThreshold", threshold=499, ref_impl=1, flavour=1),
    "edge_left_avx2": dict(fmt="wibeth", kind="edge_left", algorithm="SimpleThreshold", threshold=499, ref_impl=0, flavour=0),
    "edge_left_naive": dict(fmt="wibeth", kind="edge_left", algorithm="SimpleThreshold", threshold=499, ref_impl=1, flavour=1),
    "edge_right_avx2": dict(fmt="wibeth", kind="edge_right", algorithm="SimpleThreshold", threshold=499, ref_impl=0, flavour=0),
    "edge_right_naive": dict(fmt="wibeth", kind="edge_right", algorithm="SimpleThreshold", threshold=499, ref_impl=1, flavour=1),
    "edge_square_naive": dict(fmt="wibeth", kind="edge", algorithm="SimpleThreshold", threshold=100, ref_impl=1, flavour=1),
    "overflow_avx2": dict(fmt="wibeth", kind="overflow", algorithm="SimpleThreshold", threshold=100, ref_impl=0, flavour=0),
    "overflow_naive": dict(fmt="wibeth", kind="overflow", algorithm="SimpleThreshold", threshold=100, ref_impl=1, flavour=1),
    "noise_simple_thr60": dict(fmt="wibeth", kind="gen", seed=1, rate=0.05, n_links=2, n_units=120, algorithm="SimpleThreshold",
                               threshold=60, ref_impl=0, flavour=0),
    "noise_simple_thr20_naive": dict(fmt="wibeth", kind="gen", seed=1, rate=0.05, n_links=2, n_units=120, algorithm="SimpleThreshold",
                                     threshold=20, ref_impl=1, flavour=1),
    "dense_simple_thr8": dict(fmt="wibeth", kind="gen", seed=4, rate=0.9, n_links=1, n_units=60, algorithm="SimpleThreshold",
                              threshold=8, ref_impl=0, flavour=0),
    "noise_absrs_thr30": dict(fmt="wibeth", kind="gen", seed=2, rate=0.05, n_links=1, n_units=100, algorithm="AbsRS", threshold=30,
                              ref_impl=2, flavour=0, rs_memory_factor=8, rs_scale_factor=5),
    "noise_stdrs_thr30": dict(fmt="wibeth", kind="gen", seed=2, rate=0.05, n_links=1, n_units=100, algorithm="StandardRS", threshold=30,
                              ref_impl=3, flavour=0, rs_memory_factor=8, rs_scale_factor=5),
    "wib2_simple_thr100": dict(fmt="wib2", kind="gen", seed=5, rate=0.05, n_links=1, n_units=300, algorithm="SimpleThreshold",
                               threshold=100, ref_impl=0, flavour=0),
    "wib2_absrs_thr60": dict(fmt="wib2", kind="gen", seed=5, rate=0.05, n_links=1, n_units=300, algorithm="AbsRS", threshold=60, ref_impl=3,
                             flavour=0),
    "wib2_absrs_thr5_dense": dict(fmt="wib2", kind="gen", seed=6, rate=0.6, n_links=1, n_units=150, algorithm="AbsRS", threshold=5, ref_impl=3,
                                  flavour=0),
    "wib2_fir_thr5": dict(fmt="wib2", kind="gen", seed=5, rate=0.05, n_links=1, n_units=300, algorithm="FIR", threshold=5, ref_impl=1,
                          flavour=0),
    # thresholds beyond the packed comparator's range (sigma * 64 * threshold > 32640 once the IQR is large): the reference's
    # _mm256_cmpgt_epi16 then sees a NEGATIVE threshold; wide noise drives sigma to its clamp of 102
    "wib2_fir_thr7_noisy": dict(fmt="wib2", kind="gen", seed=7, rate=0.3, n_links=1, n_units=200, algorithm="FIR", threshold=7, ref_impl=1,
                                flavour=0, noise_q8=40 * 256),
    "wib2_fir_thr9_noisy": dict(fmt="wib2", kind="gen", seed=8, rate=0.3, n_links=1, n_units=200, algorithm="FIR", threshold=9, ref_impl=1,
                                flavour=0, noise_q8=40 * 256),
    "wib2_fir_thr5_naive": dict(fmt="wib2", kind="gen", seed=5, rate=0.05, n_links=1, n_units=300, algorithm="FIR", threshold=5,
                                ref_impl=2, flavour=1),
}


def make_input(case: dict) -> np.ndarray:
    """[n_links, n_units, unit_bytes] uint8 for a GOLDEN_CASES entry."""
    kind = case["kind"]
    if kind == "golden":
        return golden_frames()[None]
    if kind == "edge":
        return edge_square_frames()[None]
    if kind == "overflow":
        return overflow_frames()[None]
    if kind == "pulse":
        return pulse_frames()[None]
    if kind == "edge_left":
        return edge_left_frames()[None]
    if kind == "edge_right":
        return edge_right_frames()[None]
    p = S.gen_params(case["seed"], case["rate"], **({"noise_q8": case["noise_q8"]} if "noise_q8" in case else {}))
    if case["fmt"] == "wib2":
        return S.gen_wib2_host(p, case["n_links"], case["n_units"])
    return S.gen_wibeth_host(p, case["n_links"], case["n_units"])


# ---- differential cases against the reference's own compiled code ----------------------------------------------------------
# Each run returns the oracle's outputs for one input as {name: array}. What the reference returned for that input is stored in
# tests/golden/reference_outputs.npz under "<key>__<name>" (tests/golden/record_reference_outputs.py); the tests assert the
# oracle's outputs, or the GPU's, equal to it (util.assert_same_as_reference). Reference impl codes: oracle/binding.py.
def reference_outputs():
    import os

    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_outputs.npz"))


WIBETH_DIFF = [(11, 0.02, 60), (12, 0.3, 20), (13, 0.9, 8), (14, 0.9, 0), (15, 0.05, 3)]  # seed, pulse rate, threshold
WIBETH_DIFF_IMPLS = [(0, B.REF_ETH_SIMPLE_AVX2, 0), (0, B.REF_ETH_SIMPLE_NAIVE, 1), (1, B.REF_ETH_ABSRS_AVX2, 0),
                     (2, B.REF_ETH_STDRS_AVX2, 0)]  # algorithm, reference impl, oracle flavour
ACC_LIMITS = [1, 3, 10, 50, 0, -2]
WIB2_DIFF = [(31, 0.05), (32, 0.6)]
WIB2_DIFF_IMPLS = [(0, B.REF_WIB2_SIMPLE_AVX2, 0, 100), (0, B.REF_WIB2_SIMPLE_AVX2, 0, 30), (3, B.REF_WIB2_FIR_AVX2, 0, 5),
                   (3, B.REF_WIB2_FIR_NAIVE, 1, 5), (3, B.REF_WIB2_FIR_AVX2, 0, 2), (1, B.REF_WIB2_ABSRS_AVX2, 0, 60),
                   (1, B.REF_WIB2_ABSRS_AVX2, 0, 5), (1, B.REF_WIB2_ABSRS_AVX2, 0, 1), (1, B.REF_WIB2_ABSRS_AVX2, 0, 500)]
ANY_TAPS = [([2, 5, 11, 17, 9, 4, 1], 6), ([-3, 7, 20, 31, 20, 7, -3], 6), ([1, 3, 8, 10, 8, 3, 1], 5), ([300, -700, 1200, 2000, 1200, -700, 300], 6),
            ([0, 0, 0, 64, 0, 0, 0], 6)]
LANE_PRODUCT_THRESHOLDS = (11, 40, 700)  # 102*64*11 = 71808 > 65535: lanes overflow into each other
GPU_RS_DIFF = ["AbsRS", "StandardRS"]
GPU_WIB2_DIFF = [("SimpleThreshold", 60), ("FIR", 5)]
CONFIG1_THRESHOLDS = [60, 20]


def wibeth_diff(seed, rate, thr, algo, flav):
    fr = S.gen_wibeth_host(S.gen_params(seed, rate), 1, 150)[0]
    o = B.Oracle(B.make_config(algorithm=algo, threshold=thr, rs_memory_factor=8, rs_scale_factor=5), flav)
    tps, ped, _ = o.process(fr, dump=True)
    return {"tps": tps, "pedestal": ped[:, 63, :], "accum": o.state()["accum"]}  # pedestal after every frame


def acc_limit_diff(L):
    fr = S.gen_wibeth_host(S.gen_params(21, 0.2), 1, 60)[0]
    tps, ped, _ = B.Oracle(B.make_config(threshold=25, acc_limit=L)).process(fr, dump=True)
    return {"tps": tps, "pedestal": ped[:, 63, :]}


def memory_factor_diff():
    fr = S.gen_wibeth_host(S.gen_params(22, 0.2), 1, 80)[0]
    o = B.Oracle(B.make_config(algorithm=1, threshold=30))
    o.set_memory_factor(np.where(np.arange(64) % 3 == 0, 0, 8).astype(np.uint16))
    return {"tps": o.process(fr)}


def _wib2_state(o, quartiles):
    st = o.state()
    return {"pedestal": st["pedestal"], **({"quantile25": st["quantile25"], "quantile75": st["quantile75"]} if quartiles else {})}


def wib2_diff(seed, rate, algo, flav, thr):
    sc = S.gen_wib2_host(S.gen_params(seed, rate), 1, 250)[0]
    o = B.Oracle(B.make_config(fmt="wib2", algorithm=algo, threshold=thr), flav)
    return {"tps": o.process(sc), **_wib2_state(o, algo in (1, 3))}


def taps_diff(taps, exponent, flav):
    sc = S.gen_wib2_host(S.gen_params(34, 0.5), 1, 200)[0]
    o = B.Oracle(B.make_config(fmt="wib2", algorithm=3, threshold=5, fir_taps=taps, tap_exponent=exponent), flav)
    return {"tps": o.process(sc), **_wib2_state(o, True)}


def lane_product_diff(thr):
    sc = S.gen_wib2_host(S.gen_params(33, 0.4, noise_q8=40 * 256), 1, 200)[0]  # wide noise -> sigma at its clamp of 102
    return {"tps": B.Oracle(B.make_config(fmt="wib2", algorithm=3, threshold=thr)).process(sc)}


def gpu_rs_input():
    return S.gen_wibeth_host(S.gen_params(72, 0.3), 1, 300)


def gpu_rs_diff(algorithm):
    cfg = B.make_config(algorithm=S.ALGORITHMS[algorithm], threshold=30, rs_memory_factor=8, rs_scale_factor=5)
    return {"tps": B.Oracle(cfg).process(gpu_rs_input()[0], cap=1 << 20)}


def gpu_wib2_input():
    return S.gen_wib2_host(S.gen_params(73, 0.3), 1, 600)


def gpu_wib2_diff(algorithm, thr):
    cfg = B.make_config(fmt="wib2", algorithm=S.ALGORITHMS[algorithm], threshold=thr)
    return {"tps": B.Oracle(cfg).process(gpu_wib2_input()[0], cap=1 << 20)}


def config1_input():
    return S.gen_wibeth_host(S.gen_params(1, 0.05), 1, 10000)


def config1_diff(thr):
    return {"tps": B.Oracle(B.make_config(threshold=thr)).process(config1_input()[0], cap=1 << 20)}


def taps_key(taps, exponent):
    return "taps_" + "_".join(str(t) for t in taps) + f"_exp{exponent}"


def reference_runs():
    """(key, run) of every case whose reference output tests/golden/reference_outputs.npz holds."""
    for seed, rate, thr in WIBETH_DIFF:
        for algo, impl, flav in WIBETH_DIFF_IMPLS:
            yield f"wibeth_{seed}_thr{thr}_impl{impl}", lambda a=(seed, rate, thr, algo, flav): wibeth_diff(*a)
    for L in ACC_LIMITS:
        yield f"acc_limit_{L}", lambda L=L: acc_limit_diff(L)
    yield "memory_factor_per_channel", memory_factor_diff
    for seed, rate in WIB2_DIFF:
        for algo, impl, flav, thr in WIB2_DIFF_IMPLS:
            yield f"wib2_{seed}_thr{thr}_impl{impl}", lambda a=(seed, rate, algo, flav, thr): wib2_diff(*a)
    for taps, exponent in ANY_TAPS:
        yield taps_key(taps, exponent), lambda a=(taps, exponent, 0): taps_diff(*a)
    for thr in LANE_PRODUCT_THRESHOLDS:
        yield f"lane_product_thr{thr}", lambda thr=thr: lane_product_diff(thr)
    for algorithm in GPU_RS_DIFF:
        yield f"gpu_rs_{algorithm}", lambda a=algorithm: gpu_rs_diff(a)
    for algorithm, thr in GPU_WIB2_DIFF:
        yield f"gpu_wib2_{algorithm}_thr{thr}", lambda a=(algorithm, thr): gpu_wib2_diff(*a)
    for thr in CONFIG1_THRESHOLDS:
        yield f"config1_thr{thr}", lambda thr=thr: config1_diff(thr)


"""CPU: differential test of the C restatement against the reference's own code (its headers compiled unmodified behind
oracle/ref_wrapper.cpp). What the reference returns for every input here is stored in tests/golden/reference_outputs.npz
(tests/golden/record_reference_outputs.py), so the comparison needs no reference build. The last test compares two of the
reference's processors with each other; it runs only where oracle/_ref/libswtpg_ref.so was built."""
import numpy as np
import pytest

import cases
import fdreadoutlibs_b200 as S
from oracle import binding as B
from util import assert_same_as_reference


@pytest.fixture(scope="module")
def ref():
    return cases.reference_outputs()


@pytest.mark.parametrize("seed,rate,thr", cases.WIBETH_DIFF)
@pytest.mark.parametrize("algo,impl,flav", cases.WIBETH_DIFF_IMPLS)
def test_wibeth_matches_reference(seed, rate, thr, algo, impl, flav, ref):
    """TPs, the pedestal after every frame and the final accumulators."""
    assert_same_as_reference(cases.wibeth_diff(seed, rate, thr, algo, flav), ref, f"wibeth_{seed}_thr{thr}_impl{impl}")


@pytest.mark.parametrize("L", cases.ACC_LIMITS)
def test_wibeth_accumulator_limits(L, ref):
    """AVX2 SimpleThreshold honours the configured limit, including the degenerate L <= 0 cases of SURVEY A5."""
    assert_same_as_reference(cases.acc_limit_diff(L), ref, f"acc_limit_{L}")


def test_wibeth_rs_memory_factor_per_channel(ref):
    """Collection channels get R = 0 under enable_simple_threshold_on_collection (src/wibeth/WIBEthFrameProcessor.cpp:441-450)."""
    assert_same_as_reference(cases.memory_factor_diff(), ref, "memory_factor_per_channel")


@pytest.mark.parametrize("seed,rate", cases.WIB2_DIFF)
@pytest.mark.parametrize("algo,impl,flav,thr", cases.WIB2_DIFF_IMPLS)
def test_wib2_matches_reference(seed, rate, algo, impl, flav, thr, ref):
    """TPs and the final pedestals of both register selectors; the quartiles too where the algorithm keeps them."""
    assert_same_as_reference(cases.wib2_diff(seed, rate, algo, flav, thr), ref, f"wib2_{seed}_thr{thr}_impl{impl}")


@pytest.mark.parametrize("taps,exponent", cases.ANY_TAPS)
@pytest.mark.parametrize("impl,flav", [(B.REF_WIB2_FIR_AVX2, 0)])
def test_fir_arbitrary_taps_match_reference(taps, exponent, impl, flav, ref):
    """The reference's ProcessingInfo takes any taps / exponent (its frame processor only ever passes firwin_int(7, 0.1, 64) and
    6): the oracle's multiply-add chain, its 16-bit wrapping (large taps) and the exponent-dependent clamps must follow it."""
    assert_same_as_reference(cases.taps_diff(taps, exponent, flav), ref, cases.taps_key(taps, exponent))


def test_fir_threshold_64bit_lane_product(ref):
    """SURVEY H7: `sigma * multiplier * threshold` is a 4 x int64 multiply; with a large threshold the product of one
    16-bit lane carries into its neighbour. The oracle must follow the AVX2 code there too."""
    for thr in cases.LANE_PRODUCT_THRESHOLDS:
        assert_same_as_reference(cases.lane_product_diff(thr), ref, f"lane_product_thr{thr}")


@pytest.mark.skipif(not B.reference_available(), reason="oracle/_ref/libswtpg_ref.so not built")
def test_wib2_naive_rs_is_a_different_algorithm(capfd):
    """wib2/tpg/ProcessNaiveRS.hpp:22-228 is wrapped like every other processor of the reference, but it is not a scalar twin of
    wib2/tpg/ProcessRSAVX2.hpp: float running sum with R = 0.8 and scale 2 (:31-33,:122-130), quartiles of the RUNNING SUM
    (:146-152), threshold hard-wired to 5 * sigma (:175), charge = sum of the pedestal-subtracted SAMPLE >> exponent (:179).
    So there is nothing to pin to it; this test documents by how much the two disagree on ordinary input, so that nobody
    mistakes it for a parity target (the CUDA path follows the AVX2 processor, like every production configuration)."""
    sc = S.gen_wib2_host(S.gen_params(5, 0.05), 1, 100)[0]
    avx = B.ReferenceWib2(B.REF_WIB2_ABSRS_AVX2, threshold=5).process(sc)
    naive = B.ReferenceWib2(B.REF_WIB2_ABSRS_NAIVE, threshold=5).process(sc)
    capfd.readouterr()  # the header prints "Found N hits" per call
    assert avx.size == 228 and naive.size == 202
    key = lambda t: set(zip(t["channel"].tolist(), t["time_start"].tolist()))
    assert len(key(avx) & key(naive)) == 16  # 7 % of the hits share channel and start time; none of those shares its charge
    both = {k: None for k in key(avx) & key(naive)}
    ca = {(c, t): q for c, t, q in zip(avx["channel"].tolist(), avx["time_start"].tolist(), avx["adc_integral"].tolist())}
    cn = {(c, t): q for c, t, q in zip(naive["channel"].tolist(), naive["time_start"].tolist(), naive["adc_integral"].tolist())}
    assert all(ca[k] != cn[k] for k in both)

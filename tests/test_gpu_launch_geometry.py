"""GPU (B200): the launch geometries production runs, every link against the oracle.

The launch layer picks a geometry from the link count and the batch length (fdreadoutlibs_b200/csrc/swtpg_capi.cu:
launch, launch_wibeth, launch_wibeth_geo, launch_wibeth_quad, launch_wib2): 16 or 20 persistent warps per SM,
whole links or every link handed out in halving slices, the CTA form with dynamic quad claims for FIR + IQR, persistent WIB2
CTAs whose producer warp claims further links from the cursor. Each case below is sized from the device's SM count so that it
lands in one of those regimes (the headline one: pipelined SimpleThreshold, 20 warps per SM, 4 halving slices, 40 links per
SM, state carried from launch to launch), asserts that it does through `expected_geometry`, and then compares EVERY link with
the CPU oracle: its TPs, its carried state, and the number of units the launches processed.

Frames are generated on the device; launch k reads units [k * stride, (k + 1) * stride) of every link, so state crosses
launches on fresh frames. The generator is counter-based, so each oracle worker generates its own link's units on the host
and replays the same launch sequence (one `Oracle` per link, in a thread pool: ctypes releases the GIL)."""
import os
import re
import time

import numpy as np
import pytest

import fdreadoutlibs_b200 as S
from fdreadoutlibs_b200 import frames as F
from util import (FULL_WARPS_PER_SM, HIT_MIX, MAX_CTAS_PER_SM, QUAD_CTAS_PER_SM, assert_same_state, assert_same_tps, configured_oracles,
                  expected_geometry, gpu, halving_slices, ragged_units, replay_oracles, run_device, sms)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "fdreadoutlibs_b200", "csrc")

TS0 = 1 << 40  # the generator's first timestamp; a WIBEth unit spans 2048 clock ticks, a WIB2 superchunk 12 x 32
WIDE_PULSES = dict(amp_min=3000, amp_max=15000, hw_min=6, hw_max=16, ped_base=300, ped_step=3, noise_q8=40 * 256)


# ---- the launch rules util.py restates --------------------------------------------------------------------------------------
def test_restated_launch_rules_match_the_policy_constants():
    """CPU: the source lines `expected_geometry` restates. If one of them changes, update the restatement (and the cases)."""
    capi = re.sub(r"\s+", " ", open(os.path.join(CSRC, "swtpg_capi.cu")).read())
    kern = re.sub(r"\s+", " ", open(os.path.join(CSRC, "swtpg_kernels.cuh")).read())
    for line in ("constexpr auto k = wibeth_kernel<Algo, DUMP>;",
                 "const bool full_load = Algo::kFullLoadWarpsPerSm > 0 && "
                 "kp.n_links >= Algo::kFullLoadWarpsPerSm * sms + Algo::kFullLoadExtraLinks;",
                 "const unsigned warps_per_sm = full_load ? Algo::kFullLoadWarpsPerSm : Algo::kWarpsPerSm;",
                 "unsigned even = per_sm >= 4 ? per_sm / 4 * 4 : per_sm;",
                 "if (warps_per_sm > 0) // the measured optimum, if the device holds that many even = std::min(even, warps_per_sm);",
                 "const unsigned grid = std::min<unsigned>(std::min<unsigned>(kp.n_links, even * sms), resident);",
                 "if (kp.n_links > grid && (full_load || kp.n_links % grid != 0))",
                 "parts = std::max(1u, std::min(4u, kp.units_stride / 16u));",
                 "kq.slice_geom = 1u; // halving slices",
                 "if constexpr (Algo::kQuadCtasPerSm > 0) return launch_wibeth_quad<Algo, DUMP>(kp, s); "
                 "else return launch_wibeth_geo<Algo, DUMP>(kp, s);",
                 "case Policy::WibEthSimple: return launch_wibeth<PackedSimpleWibEthPipe, DUMP>(kp, s);",
                 "case Policy::WibEthAbsRs: return launch_wibeth<PackedRsWibEth<false>, DUMP>(kp, s);",
                 "case Policy::WibEthStandardRs: return launch_wibeth<PackedRsWibEth<true>, DUMP>(kp, s);"):
        assert line in capi, f"swtpg_capi.cu no longer has `{line}`"
    for line in (# ScalarAlgo: as many warps as fit, never full load
                 "static constexpr int kWarpsPerSm = 0; static constexpr int kFullLoadWarpsPerSm = 0; "
                 "static constexpr int kFullLoadExtraLinks = 0; static constexpr int kQuadCtasPerSm = 0;",
                 # PackedSimpleT (the pipelined form) runs the one-warp-per-CTA form: 16 per SM, from 20 * SMs links on 20
                 f"static constexpr int kWarpsPerSm = 16; static constexpr int kFullLoadWarpsPerSm = {FULL_WARPS_PER_SM}; "
                 "static constexpr int kFullLoadExtraLinks = 0; static constexpr int kQuadCtasPerSm = 0;",
                 # PackedRsWibEth (derives from PackedSimpleT): its own warps, full load from 20 * SMs + 1 links on
                 "static constexpr int kWarpsPerSm = STANDARD ? 20 : 16; static constexpr int kFullLoadExtraLinks = 1;",
                 "struct PackedRsWibEth : PackedSimpleWibEth",
                 # the halving slices halving_slices restates
                 "u0 = n - ((n + (1u << part) - 1u) >> part); "
                 "u1 = part + 1u == (1u << p.parts_log2) ? n : n - ((n + (2u << part) - 1u) >> (part + 1u));"):
        assert line in kern, f"swtpg_kernels.cuh no longer has `{line}`"
    assert kern.count(f"static constexpr int kQuadCtasPerSm = {QUAD_CTAS_PER_SM};") == 2  # PackedFirIqr, PackedFirIqrAnyTaps
    # the restatement itself at B200's 148 SMs, for the regimes the GPU cases rely on
    assert expected_geometry("SimpleThreshold", 40 * 148, 64, 148) == (20, 4)
    assert expected_geometry("SimpleThreshold", 20 * 148, 64, 148) == (20, 1)
    assert expected_geometry("SimpleThreshold", 20 * 148 + 1, 100, 148) == (20, 4)
    assert expected_geometry("SimpleThreshold", 20 * 148 - 1, 64, 148) == (16, 4)
    assert expected_geometry("SimpleThreshold", 16 * 148 + 1, 48, 148) == (16, 2)
    assert expected_geometry("SimpleThreshold", 32 * 148, 64, 148) == (20, 4)
    assert expected_geometry("SimpleThreshold", 16 * 148, 64, 148) == (16, 1)
    assert expected_geometry("AbsRS", 20 * 148, 64, 148) == (16, 4)
    assert expected_geometry("AbsRS", 16 * 148, 64, 148) == (16, 1)  # one whole round of its own 16 per SM: whole links
    assert expected_geometry("AbsRS", 20 * 148 + 1, 64, 148) == (20, 4)
    assert expected_geometry("StandardRS", 20 * 148, 64, 148) == (20, 1)
    assert expected_geometry("StandardRS", 40 * 148, 16, 148) == (20, 1)
    assert [expected_geometry("scalar", 32 * 148 + 1, 64, 148, f)[1] for f in range(1, 33)] == [4] * 32
    assert halving_slices(100, 4) == [(0, 50), (50, 75), (75, 87), (87, 100)]
    assert halving_slices(3, 4) == [(0, 1), (1, 2), (2, 2), (2, 3)]


# ---- harness --------------------------------------------------------------------------------------------------------------
def locate(tp, fmt: str, stride: int, nus, slices: int) -> str:
    """Launch, unit and slice a TP's start falls in (for the failure message)."""
    unit = (int(tp["time_start"]) - TS0) // (384 if fmt == "wib2" else 2048)
    k, u = divmod(unit, stride)
    if k >= len(nus):
        return f"unit {unit} (after the last launch)"
    n = stride if nus[k] is None else int(nus[k][int(tp["link"])])
    part = next((p for p, (u0, u1) in enumerate(halving_slices(n, slices)) if u0 <= u < u1), None)
    return f"launch {k}, unit {u} of {n}, slice {part} of {slices}"


def check_every_link(what, fmt, algorithm, n_links, stride, nus, seed, rate, thr, slices=1, tp_capacity=1 << 24, rs_factors=None,
                     gen_kw=None, oracle_cap=1 << 18, min_tps=1, **kw):
    """Runs the launches on the GPU and the oracle, then compares every link: TPs, carried state, units processed."""
    p = S.gen_params(seed, rate, **(gen_kw or {}))
    handle = dict(algorithm=algorithm, threshold=thr, **kw)
    t0 = time.time()
    got, gstate, _ = run_device(fmt, n_links, stride, nus, p, rs_factors=rs_factors, tp_capacity=tp_capacity, **handle)
    t1 = time.time()
    oracle_of = configured_oracles(fmt, handle, rs_tables=None if rs_factors is None else dict(enumerate(rs_factors)))
    want, ostate = replay_oracles(fmt, n_links, stride, nus, p, oracle_of, cap=oracle_cap)
    t2 = time.time()

    allg = np.concatenate(got)
    assert allg.size >= min_tps, f"{what}: only {allg.size} TPs, the case does not exercise the hit path"
    assert allg.size == 0 or int(allg["link"].max()) < n_links
    allg = allg[np.argsort(allg["link"], kind="stable")]
    bounds = np.searchsorted(allg["link"], np.arange(n_links + 1))
    for l in range(n_links):
        mine, theirs = F.sort_tps(allg[bounds[l]:bounds[l + 1]]), F.sort_tps(want[l])
        if mine.size == theirs.size and (mine == theirs).all():
            continue
        if mine.size == theirs.size:
            first = mine[np.nonzero(mine != theirs)[0][0]]
        else:  # the first record one side has and the other lacks
            a, b = set(mine.tolist()), set(theirs.tolist())
            first = np.array([min((a ^ b), key=lambda r: (r[0], r[6], r[5]))], dtype=F.TP_DTYPE)[0]
        assert_same_tps(mine, theirs, f"{what}: link {l} ({locate(first, fmt, stride, nus, slices)})")
    assert_same_state(gstate, ostate, fmt, algorithm, what)
    print(f"{what}: {n_links} links, {allg.size} TPs identical; GPU {t1 - t0:.1f} s, oracle {t2 - t1:.1f} s")


# ---- WIBEth, one warp per CTA -----------------------------------------------------------------------------------------------
@gpu
def test_full_load_whole_rounds():
    """The bench's input and geometry, the headline number's: pipelined SimpleThreshold, 40 links per SM = two whole rounds of
    20 warps per SM, every link in 4 halving slices, two launches with the state carried from one to the next."""
    n = 40 * sms()
    assert expected_geometry("SimpleThreshold", n, 64, sms()) == (20, 4)
    check_every_link("full load", "wibeth", "SimpleThreshold", n, 64, [None, None], seed=2, rate=0.02, thr=60, slices=4, min_tps=100000)


@gpu
def test_full_load_device_ordered():
    """The same launch with SWTPG_FLAG_SORTED_TPS: the device-ordered list equals the host order of the plain list record for
    record, with nothing finished on the host. Link numbers up to 40 * SMs need a 13-bit link key. The plain list of this
    input is the first launch of test_full_load_whole_rounds, checked there against the oracle link for link."""
    n = 40 * sms()
    p = S.gen_params(2, 0.02)
    plain, _, _ = run_device("wibeth", n, 64, [None], p, tp_capacity=1 << 22, threshold=60)
    ordered, _, info = run_device("wibeth", n, 64, [None], p, tp_capacity=1 << 22, threshold=60, sorted_tps=True)
    want = S.sort_tps(plain[0])
    assert want.size > 100000 and int(want["link"].max()) >= 4096
    assert ordered[0].size == want.size and (ordered[0] == want).all()
    assert info["sort"]["lists"] == 1 and info["sort"]["finished_on_host"] == 0


@gpu
def test_full_load_tail():
    """One link more than a round of 20 warps per SM, 100 units: slices of 50 / 25 / 12 / 13 units and a one-link tail round."""
    n = 20 * sms() + 1
    assert expected_geometry("SimpleThreshold", n, 100, sms()) == (20, 4)
    assert [u1 - u0 for u0, u1 in halving_slices(100, 4)] == [50, 25, 12, 13]
    check_every_link("full-load tail", "wibeth", "SimpleThreshold", n, 100, [None, None], seed=101, rate=0.3, thr=30, slices=4)


@gpu
def test_one_round_exactly():
    """The boundary itself: exactly one link per warp of the 20-per-SM grid keeps whole links."""
    n = 20 * sms()
    assert expected_geometry("SimpleThreshold", n, 64, sms()) == (20, 1)
    check_every_link("one round", "wibeth", "SimpleThreshold", n, 64, [None], seed=102, rate=0.1, thr=60)


@gpu
def test_partial_load():
    """Below the full-load boundary (16 warps per SM) and not a whole number of rounds: 48 units = 2 slices of 24."""
    n = 16 * sms() + 1
    assert expected_geometry("SimpleThreshold", n, 48, sms()) == (16, 2)
    check_every_link("partial load", "wibeth", "SimpleThreshold", n, 48, [None, None], seed=103, rate=0.2, thr=25, slices=2)


@gpu
def test_ragged_production_shape():
    """The headline geometry with ragged unit counts around every slice edge (empty slices, fewer units than slices, empty
    links), then an all-empty launch, then a full one: the per-link slice counters and the cursor re-arm after each."""
    n = 40 * sms()
    assert expected_geometry("SimpleThreshold", n, 64, sms()) == (20, 4)
    nus = [ragged_units(104, n, 64, HIT_MIX), np.zeros(n, dtype=np.uint32), None]
    check_every_link("ragged", "wibeth", "SimpleThreshold", n, 64, nus, seed=104, rate=0.2, thr=30, slices=4)


@gpu
def test_dense_hits_across_slices():
    """The bench's stress input (threshold 8, 0.5 pulses per channel and frame) in 4 slices: the hit staging is flushed at
    every slice end while hits are open across the slice boundaries; about 11 k TPs per link."""
    n = 20 * sms() + 1
    assert expected_geometry("SimpleThreshold", n, 64, sms()) == (20, 4)
    check_every_link("dense hits", "wibeth", "SimpleThreshold", n, 64, [None], seed=105, rate=0.5, thr=8, slices=4,
                     tp_capacity=1 << 26, oracle_cap=1 << 16, min_tps=10_000_000)


@gpu
def test_abs_rs_partial_load_with_memory_factors():
    """AbsRS below one 20-per-SM round (its own 16 warps per SM), not whole rounds: 4 slices; per-channel memory factors 0..12
    (about 14 k TPs per link and launch)."""
    n = 16 * sms() + 1
    assert expected_geometry("AbsRS", n, 64, sms()) == (16, 4)
    factors = np.random.default_rng(106).integers(0, 13, (n, 64)).astype(np.uint16)
    factors[:, 0] = 0
    check_every_link("AbsRS partial load", "wibeth", "AbsRS", n, 64, [None, None], seed=106, rate=0.2, thr=30, slices=4,
                     rs_factors=factors, rs_memory_factor=8, rs_scale_factor=5, tp_capacity=1 << 26, oracle_cap=1 << 16)


@gpu
def test_abs_rs_full_load():
    n = 40 * sms()
    assert expected_geometry("AbsRS", n, 64, sms()) == (20, 4)
    check_every_link("AbsRS full load", "wibeth", "AbsRS", n, 64, [None], seed=107, rate=0.2, thr=30, slices=4)


@gpu
def test_standard_rs_full_load():
    n = 20 * sms() + 1
    assert expected_geometry("StandardRS", n, 64, sms()) == (20, 4)
    check_every_link("StandardRS full load", "wibeth", "StandardRS", n, 64, [None, None], seed=108, rate=0.2, thr=30, slices=4,
                     rs_memory_factor=7, rs_scale_factor=2)


@gpu
@pytest.mark.parametrize("algorithm,thr,kw", [("SimpleThreshold", 30, dict(acc_limit=0)), ("FIR", 5, dict(tap_exponent=11))],
                         ids=["simple_acc_limit_0", "fir_exponent_11"])
def test_scalar_fallback_sliced(algorithm, thr, kw):
    """The scalar policies (ScalarAlgo) run as many warps as fit, at most 32 single-warp CTAs per SM, so 32 * SMs + 1 links are
    sliced at any occupancy. For FIR the ring phase is carried across the slice boundaries."""
    n = 32 * sms() + 1
    assert {expected_geometry("scalar", n, 64, sms(), fits)[1] for fits in range(1, MAX_CTAS_PER_SM + 1)} == {4}
    check_every_link(f"scalar {algorithm} sliced", "wibeth", algorithm, n, 64, [None, None], seed=109, rate=0.2, thr=thr, slices=4, **kw)


@gpu
@pytest.mark.parametrize("fmt,algorithm,thr,kw", [
    ("wibeth", "AbsRS", 30, dict(acc_limit=0)), ("wibeth", "StandardRS", 30, dict(acc_limit=0, rs_memory_factor=7, rs_scale_factor=2)),
    ("wib2", "FIR", 5, dict(tap_exponent=11)), ("wib2", "AbsRS", 5, dict(tap_exponent=11, gen_kw=WIDE_PULSES))])
def test_scalar_policies_of_the_launch_table(fmt, algorithm, thr, kw):
    """ScalarAlgo instantiations of launch() that no other test selects: the running sums with accumulator limit 0, and WIB2
    FIR / AbsRS with a tap exponent beyond the packed policies' range (AbsRS finds hits there only on pulses of up to the
    full 14-bit range). Ragged batches, three launches."""
    n = 40 if fmt == "wibeth" else 9
    nus = [ragged_units(110 + k, n, 16, (0, 1, 16)) for k in range(3)]
    check_every_link(f"scalar {fmt} {algorithm}", fmt, algorithm, n, 16, nus, seed=110, rate=0.4, thr=thr, **kw)


# ---- CTA forms --------------------------------------------------------------------------------------------------------------
ANY_TAPS_1 = ([-3, 7, 20, 31, 20, 7, -3], 6)  # test_gpu_parity.py ANY_TAPS[1]: PackedFirIqrAnyTaps


@gpu
@pytest.mark.parametrize("taps", [None, ANY_TAPS_1], ids=["firwin", "any_taps"])
def test_fir_quads_claimed_after_the_first_round(taps):
    """FIR + IQR runs the CTA form: persistent CTAs of 4 link-warps claim quads of links; 16 * SMs + 3 links are one quad more
    than the first round, and the last quad has 3 links."""
    n = 16 * sms() + 3
    assert (n + 3) // 4 == QUAD_CTAS_PER_SM * sms() + 1 and n % 4 == 3
    kw = {} if taps is None else dict(fir_taps=taps[0], tap_exponent=taps[1])
    nus = [ragged_units(111 + k, n, 16, (0, 1, 16)) for k in range(2)]
    check_every_link("FIR quads", "wibeth", "FIR", n, 16, nus, seed=111, rate=0.3, thr=5, **kw)


WIB2_MAX_CTAS_PER_SM = 6  # wib2_kernel: about 35.6 KB of shared memory and 160 threads per CTA


@gpu
@pytest.mark.parametrize("algorithm,thr", [("SimpleThreshold", 60), ("FIR", 5), ("AbsRS", 60)])
def test_wib2_ctas_take_several_links(algorithm, thr):
    """WIB2: at most 6 persistent CTAs per SM, so 20 * SMs links give every CTA several links, claimed by its producer warp
    from the cursor and handed to the consumer warps through the link FIFO; ragged unit counts include empty links."""
    n = 20 * sms()
    assert n > 3 * WIB2_MAX_CTAS_PER_SM * sms()
    nus = [ragged_units(112 + k, n, 16, (0, 1, 16)) for k in range(2)]
    check_every_link(f"WIB2 {algorithm}", "wib2", algorithm, n, 16, nus, seed=112, rate=0.3, thr=thr)

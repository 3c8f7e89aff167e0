"""GPU (B200): the launch geometries production runs, every link against the oracle.

The launch layer picks a geometry from the link count and the batch length (fdreadoutlibs_b200/csrc/swtpg_capi.cu:
launch_wibeth_geo, launch_wibeth_simple, launch_wibeth, launch_wibeth_quad, launch_wib2): 16 or 20 persistent warps per SM,
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
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import fdreadoutlibs_b200 as S
from fdreadoutlibs_b200 import frames as F
from oracle import binding as B
from util import assert_same_tps

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "fdreadoutlibs_b200", "csrc")

# Tuning aids change the geometry a launch takes, so under any of them the regimes asserted below are not the ones that run.
TUNING_AIDS = ("SWTPG_PARTS", "SWTPG_WARPS", "SWTPG_SIMPLE_PIPE", "SWTPG_CTAS_PER_SM", "SWTPG_WIBETH_KERNEL", "SWTPG_SLICE_GEOM",
               "SWTPG_FORCE_SCALAR", "SWTPG_LIB")


def gpu(test):
    skip = pytest.mark.skipif(any(v in os.environ for v in TUNING_AIDS), reason="a tuning aid is set: launches leave the default geometry")
    return pytest.mark.gpu(skip(test))


TS0 = 1 << 40  # the generator's first timestamp; a WIBEth unit spans 2048 clock ticks, a WIB2 superchunk 12 x 32
WIDE_PULSES = dict(amp_min=3000, amp_max=15000, hw_min=6, hw_max=16, ped_base=300, ped_step=3, noise_q8=40 * 256)
HIT_MIX = (0, 1, 2, 3, 4, 5, 7, 8, 9, 15, 16, 17, 31, 32, 33, 63, 64)  # unit counts around every slice edge of stride 64


# ---- the launch rules, restated -------------------------------------------------------------------------------------------
# swtpg_capi.cu:100-135 (launch_wibeth_geo), :197-241 (launch_wibeth_simple, launch_wibeth), and the policies' constants
# kWarpsPerSm / kQuadCtasPerSm (swtpg_kernels.cuh:476, 816, 979-981, 1381). test_restated_rules_match_the_source pins the
# source lines this depends on, so the table has to be updated together with the rules.
FULL_WARPS_PER_SM = 20   # kFullWarpsPerSm, and the running sums' 20 warps per SM above one round
QUAD_CTAS_PER_SM = 4     # PackedFirIqr / PackedFirIqrAnyTaps::kQuadCtasPerSm
MAX_CTAS_PER_SM = 32     # what an sm_100 SM holds at most


def expected_geometry(policy: str, n_links: int, units_stride: int, sms: int, fits: int = MAX_CTAS_PER_SM):
    """(persistent warps per SM, slices per link) of a WIBEth launch of the one-warp-per-CTA form. `fits`: single-warp CTAs of
    the policy an SM holds (occupancy); every packed policy fits at least the 20 it asks for. policy: "SimpleThreshold"
    (the pipelined form every packed launch runs), "AbsRS", "StandardRS", "scalar" (ScalarAlgo: as many warps as fit)."""
    even = fits // 4 * 4 if fits >= 4 else fits  # a multiple of 4: every SM sub-partition loaded alike
    if policy == "SimpleThreshold":  # PackedSimpleWibEthPipe: 16 per SM, from 20 * SMs links on 20 and slices for whole rounds
        cap, whole_rounds = (FULL_WARPS_PER_SM, True) if n_links >= FULL_WARPS_PER_SM * sms else (16, False)
    elif policy in ("AbsRS", "StandardRS"):  # PackedRsWibEth: 16 (AbsRS) / 20 (StandardRS), above one 20-per-SM round 20, sliced
        cap, whole_rounds = (FULL_WARPS_PER_SM, True) if n_links > FULL_WARPS_PER_SM * sms else (16 if policy == "AbsRS" else 20, False)
    elif policy == "scalar":
        cap, whole_rounds = even, False
    else:
        raise ValueError(policy)
    warps = min(even, cap)
    persistent = min(n_links, warps * sms)
    parts = 1
    if n_links > persistent and (whole_rounds or n_links % persistent != 0):
        parts = max(1, min(4, units_stride // 16))
    return warps, 1 << (parts.bit_length() - 1)  # the largest power of two not above it


def halving_slices(n: int, slices: int):
    """[u0, u1) of each slice of a link with n units (SWTPG_AUTO_SLICE_GEOM = 1; tests/test_slice_arithmetic.py pins it)."""
    out = []
    for part in range(slices):
        u0 = n - ((n + (1 << part) - 1) >> part)
        u1 = n if part + 1 == slices else n - ((n + (2 << part) - 1) >> (part + 1))
        out.append((u0, u1))
    return out


def test_restated_rules_match_the_source():
    """CPU: the source lines `expected_geometry` restates. If one of them changes, update the restatement (and the cases)."""
    capi = re.sub(r"\s+", " ", open(os.path.join(CSRC, "swtpg_capi.cu")).read())
    kern = re.sub(r"\s+", " ", open(os.path.join(CSRC, "swtpg_kernels.cuh")).read())
    for line in ("#define SWTPG_AUTO_SLICE_GEOM 1",
                 "unsigned even = G::warps == 1 && per_sm >= 4 ? per_sm / 4 * 4 : per_sm;",
                 "even = std::min<unsigned>(even, unsigned(kWarpsPerSm));",
                 "if (kp.n_links > persistent && (SLICE_WHOLE_ROUNDS || kp.n_links % persistent != 0))",
                 "parts = std::max(1u, std::min(4u, kp.units_stride / 16u));",
                 f"constexpr int kFullWarpsPerSm = {FULL_WARPS_PER_SM};",
                 "if (kp.n_links >= unsigned(kFullWarpsPerSm * sms))",
                 "return launch_wibeth_geo<PackedSimpleWibEthPipe, DUMP, GeoDefault, kFullWarpsPerSm, true>(kp, s);",
                 "return launch_wibeth_geo<PackedSimpleWibEthPipe, DUMP, GeoDefault>(kp, s); }",
                 f"if (kp.n_links > unsigned({FULL_WARPS_PER_SM} * sms)) return launch_wibeth_geo<Algo, DUMP, GeoDefault, {FULL_WARPS_PER_SM}, true>(kp, s);"):
        assert line in capi, f"swtpg_capi.cu no longer has `{line}`"
    for line in ("static constexpr int kWarpsPerSm = PIPE ? 16 : 20;", "static constexpr int kWarpsPerSm = STANDARD ? 20 : 16;",
                 "static constexpr int kWarpsPerSm = 0;", "#define SWTPG_QUAD_SIMPLE 0"):
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
def sms() -> int:
    import torch

    return torch.cuda.get_device_properties(0).multi_processor_count


BASE_FIELDS = ["pedestal", "accum", "prev_was_over", "hit_charge", "hit_tover", "initialized"]


def state_fields(fmt: str, algorithm: str):
    """The carried state each policy keeps (as test_gpu_parity.py's oracle tests compare it)."""
    f = list(BASE_FIELDS)
    if fmt == "wibeth" and algorithm != "FIR":
        f += ["hit_peak_adc", "hit_peak_time"]
    if fmt == "wibeth" and algorithm in ("AbsRS", "StandardRS"):
        f += ["rs", "pedestal_rs", "accum_rs", "rs_memory_factor"]
    if algorithm == "FIR":
        f += ["quantile25", "quantile75", "accum25", "accum75", "prev_samp"]
    return f


def ragged_units(seed: int, n_links: int, stride: int, specials=()):
    """Seeded per-link unit counts in [0, stride], with each of `specials` on a few links spread over the whole range."""
    rng = np.random.default_rng(seed)
    nu = rng.integers(0, stride + 1, n_links).astype(np.uint32)
    specials = [s for s in specials if s <= stride]
    at = rng.choice(n_links, size=min(n_links, 4 * len(specials)), replace=False)
    for i, l in enumerate(at):
        nu[l] = specials[i % len(specials)]
    return nu


def locate(tp, fmt: str, stride: int, nus, slices: int) -> str:
    """Launch, unit and slice a TP's start falls in (for the failure message)."""
    unit = (int(tp["time_start"]) - TS0) // (384 if fmt == "wib2" else 2048)
    k, u = divmod(unit, stride)
    if k >= len(nus):
        return f"unit {unit} (after the last launch)"
    n = stride if nus[k] is None else int(nus[k][int(tp["link"])])
    part = next((p for p, (u0, u1) in enumerate(halving_slices(n, slices)) if u0 <= u < u1), None)
    return f"launch {k}, unit {u} of {n}, slice {part} of {slices}"


def run_gpu(fmt, n_links, stride, nus, p, tp_capacity, rs_factors=None, **handle_kw):
    """Every launch of one handle on device-generated frames: (TP list of each launch, per-link state, counters [+ sort stats])."""
    import torch

    unit_bytes = F.WIB2_SUPERCHUNK_BYTES if fmt == "wib2" else F.WIBETH_FRAME_BYTES
    gen = S.gen_wib2_device if fmt == "wib2" else S.gen_wibeth_device
    buf = torch.empty(n_links * stride * unit_bytes, dtype=torch.uint8, device="cuda")
    got = []
    try:
        with S.TPGenerator(n_links, stride, fmt=fmt, tp_capacity=tp_capacity, **handle_kw) as g:
            if rs_factors is not None:
                g.set_rs_memory_factor(rs_factors)
            g.start()
            for k, nu in enumerate(nus):
                gen(p, buf.data_ptr(), n_links, stride, unit0=k * stride)
                torch.cuda.synchronize()  # the generator runs on the legacy stream, the handle on its own
                g.process_device(buf.data_ptr(), stride, n_units=nu)
                got.append(g.fetch_tps(cap=tp_capacity))  # waits for the launch: the buffer is free to be rewritten
            states = np.stack([g.dump_state(l) for l in range(n_links)])
            info = g.counters()
            if handle_kw.get("sorted_tps"):
                info["sort"] = g.sort_stats()
    finally:
        del buf
        torch.cuda.empty_cache()
    return got, states, info


def run_oracle(cfg, fmt, n_links, stride, nus, p, rs_factors=None, cap=1 << 18):
    """The same launch sequence per link on the CPU: (TPs of each link, per-link state)."""
    gen = S.gen_wib2_host if fmt == "wib2" else S.gen_wibeth_host

    def one(l):
        o = B.Oracle(cfg, link_id=l)
        if rs_factors is not None:
            o.set_memory_factor(rs_factors[l])
        parts = []
        for k, nu in enumerate(nus):
            n = stride if nu is None else int(nu[l])
            if n:
                parts.append(o.process(gen(p, 1, n, link0=l, unit0=k * stride, n_threads=1)[0], cap=cap))
        return np.concatenate(parts) if parts else np.zeros(0, dtype=F.TP_DTYPE), o.state()

    with ThreadPoolExecutor(os.cpu_count() or 1) as ex:
        res = list(ex.map(one, range(n_links)))
    return [r[0] for r in res], np.stack([r[1] for r in res])


def check_every_link(what, fmt, algorithm, n_links, stride, nus, seed, rate, thr, slices=1, tp_capacity=1 << 24, rs_factors=None,
                     gen_kw=None, oracle_cap=1 << 18, min_tps=1, **kw):
    """Runs the launches on the GPU and the oracle, then compares every link: TPs, carried state, units processed."""
    p = S.gen_params(seed, rate, **(gen_kw or {}))
    t0 = time.time()
    got, gstate, info = run_gpu(fmt, n_links, stride, nus, p, tp_capacity, rs_factors, algorithm=algorithm, threshold=thr, **kw)
    t1 = time.time()
    okw = {k: v for k, v in kw.items() if k in ("acc_limit", "rs_memory_factor", "rs_scale_factor", "fir_taps", "tap_exponent")}
    cfg = B.make_config(fmt=fmt, algorithm=S.ALGORITHMS[algorithm], threshold=thr, **okw)
    want, ostate = run_oracle(cfg, fmt, n_links, stride, nus, p, rs_factors, oracle_cap)
    t2 = time.time()

    assert info["units_processed"] == sum(n_links * stride if nu is None else int(nu.sum()) for nu in nus), \
        f"{what}: {info['units_processed']} units processed"
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
    for f in state_fields(fmt, algorithm):
        bad = (gstate[f] != ostate[f]).reshape(n_links, -1).any(axis=1)
        if bad.any():
            l = int(np.nonzero(bad)[0][0])
            ch = int(np.nonzero((gstate[f][l] != ostate[f][l]).reshape(gstate.shape[1], -1).any(axis=1))[0][0])
            pytest.fail(f"{what}: state field {f} differs on {int(bad.sum())} links, first link {l} channel {ch}: "
                        f"GPU {gstate[f][l][ch]}, oracle {ostate[f][l][ch]}")
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
    plain, _, _ = run_gpu("wibeth", n, 64, [None], p, 1 << 22, threshold=60)
    ordered, _, info = run_gpu("wibeth", n, 64, [None], p, 1 << 22, threshold=60, sorted_tps=True)
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
